#!/usr/bin/env python
"""Headline benchmark: ST-encoder fbank frames/s (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg2|cfg1]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one synthetic batch: per-utterance fbank CMVN, then the
encoder forward (conv subsampling -> 11 pre-LN layers with log-penalty attention -> CTC argmax
compression at layer 8 -> final LN).  Workload at N=1 = BASELINE.json configs[1] (EACL'21 encoder,
d512 h8 ffn2048, bf16, batch 64 x 1500 x 40).  For N>1 the path shards by utterance batch: every rank
runs its own batch, no collective on the data path (scaling "weak").

Prints ONE JSON line (rank 0).  Keys: see the bench contract in the task statement.
`value`: K steps back to back through `EncoderPipeline.run_device` (batches resident in HBM, two
forwards in flight on two compute lanes), one CUDA-event pair around all K steps, max over ranks.
`e2e`: the same K steps through `EncoderPipeline.run` from pinned HOST buffers (H2D of every batch and
D2H of every result inside the timed wall-clock region).  `single_forward_ms`: one forward at a time with
an L2 flush before each (informative).  `roofline`: dominant kernel family (the tcgen05 linear kernel),
timed live with CUDA events in a separate launch-by-launch pass; `kernels`: the same pass for every
kernel family; `cpu_baseline`: the oracle port on the host cores (rank 0, bounded sample).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "fbk-fairseq-st_b200"))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

CONFIGS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on
    "cfg2": dict(model=dict(embed_dim=512, ffn_dim=2048, heads=8, layers=11, conv_channels=64,
                            feat_dim=40, vocab=8005, distance_penalty="log", ctc_layer=8,
                            ctc_strategy="avg"),
                 lengths=[1500] * 64,
                 name="EACL21 CTC-compression ST encoder: 11L d512 h8 ffn2048, log penalty, "
                      "ctc-compress avg @8, batch 64x1500x40"),
    # BASELINE.json configs[0]: the reference's own CPU-runnable case
    "cfg1": dict(model=dict(embed_dim=256, ffn_dim=768, heads=4, layers=6, conv_channels=64,
                            feat_dim=40, vocab=105, distance_penalty=None, ctc_layer=4,
                            ctc_strategy="avg"),
                 lengths=[1000, 950, 900, 800, 700, 600, 500, 400],
                 name="6L d256 h4 ffn768, ctc-compress avg @4, batch 8x1000x40"),
    # BASELINE.json configs[2] (one length bucket of it; informative, not the headline line):
    # ragged utterances of one bucket (sorted by length, ~96 k frames per GPU), weighted pooling
    "cfg3": dict(model=dict(embed_dim=512, ffn_dim=2048, heads=8, layers=11, conv_channels=64,
                            feat_dim=40, vocab=8005, distance_penalty="log", ctc_layer=8,
                            ctc_strategy="weighted"),
                 lengths=[2000 - 13 * i for i in range(48)],
                 name="cfg2 model, ctc-compress weighted @8, one ragged length bucket 48 x 1389..2000 x 40"),
    # BASELINE.json configs[4]: long-form stress (conv_transformer_giant: C=128, conv_transformer.py:565)
    "cfg5": dict(model=dict(embed_dim=1024, ffn_dim=4096, heads=16, layers=12, conv_channels=128,
                            feat_dim=80, vocab=8005, distance_penalty="log", ctc_layer=8,
                            ctc_strategy="avg"),
                 lengths=[6000, 5600, 5200, 4800, 4400, 4000, 3500, 3000],
                 name="long-form 12L d1024 h16 ffn4096 C128, ctc-compress avg @8, batch 8 x 3000..6000 x 80"),
}
# BASELINE.json configs[3]: full ST training step -- the cfg2 encoder + a 6-layer decoder, joint CTC +
# label-smoothed CE, bf16, NCCL gradient all-reduce (bench.py --config cfg4; see run_train)
CONFIGS["cfg4"] = dict(model=CONFIGS["cfg2"]["model"], lengths=[1500] * 64,
                       decoder=dict(layers=6, tgt_vocab=8000, tgt_len=64, transcript_len=48),
                       name="EACL21 ST training step: cfg2 encoder (11L d512, log penalty, ctc-compress avg @8) + "
                            "6-layer d512 decoder, ctc_multi_loss (CTC + label-smoothed CE), batch 64x1500x40 per GPU")
CTC_MARGIN = 30.0
LOOKAHEAD_CYCLES = int(1.0e-3 * 1.9e9)  # ~1 ms of untimed GPU delay before every timed step
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full`
# captures (profiles/r01i_ncu_gemm2.txt: mean over the captured launches of each kernel: qkv + fc1,
# out_proj + fc2 of a full-length layer; cold caches, so an upper bound for the L2-warm step)
NCU_TRAFFIC = {
    "gemm2_kernel<bf16 out> (qkv, fc1, ctc_fc)": int((26.99 + 17.42 + 27.55 + 39.86) / 2 * 1e6),
    "gemm2_kernel<f32 out + residual (+ bf16 copy, LN statistics)> (out_proj, fc2)":
        int((74.31 + 23.66 + 151.59 + 35.04) / 2 * 1e6),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"],
                    src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


# ------------------------------------------------------------------------------ synthetic data
def make_batch(lengths, feat_dim, seed):
    """src_tokens ~ N(0,1)*3+1 (un-normalised fbank-like), zeroed past each length (collater
    semantics, data/collaters.py:51-56)."""
    g = torch.Generator().manual_seed(seed)
    B, T = len(lengths), max(lengths)
    x = torch.randn(B, T, feat_dim, generator=g) * 3.0 + 1.0
    for b, n in enumerate(lengths):
        x[b, n:] = 0
    return x, torch.tensor(lengths, dtype=torch.long)


def label_plan(L, B, vocab, seed, mean_run=3.0, blank_prob=0.5):
    """Run-structured CTC label plan (SURVEY F9/8d): geometric run lengths (mean 3), about a third of the
    runs are <ctc_blank>, and two adjacent runs never share a label (a blank run is followed by a
    non-blank one, a repeated label is re-drawn as its successor), so the number of segments equals
    the number of runs and the compression ratio is ~1/mean_run = 0.33 (the survey's figure).
    O(L/mean_run) vector steps over the batch."""
    g = torch.Generator().manual_seed(seed)
    p = 1.0 / mean_run
    start = torch.rand(L, B, generator=g) < p  # Bernoulli(p): "a new run starts here"
    start[0] = True
    run_id = torch.cumsum(start.long(), 0) - 1  # L x B
    n_runs = int(run_id.max()) + 1
    labs = torch.randint(4, vocab - 1, (n_runs, B), generator=g)
    want_blank = torch.rand(n_runs, B, generator=g) < blank_prob
    blank_id = vocab - 1
    prev = torch.full((B,), -1, dtype=torch.long)
    for r in range(n_runs):
        cur = torch.where(want_blank[r] & (prev != blank_id), torch.full((B,), blank_id), labs[r])
        clash = cur == prev  # a non-blank label drawn twice in a row: take the next label instead
        cur = torch.where(clash, 4 + (cur - 4 + 1) % (vocab - 5), cur)
        labs[r] = cur
        prev = cur
    return torch.gather(labs, 0, run_id)


def randomise_norm_stats(enc, seed):
    """BN running stats / affine and biases away from the identity so every epilogue term matters
    (BASELINE.md section 3)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for bn in enc.bn:
            bn.running_mean.copy_(torch.randn(bn.running_mean.shape, generator=g) * 0.1)
            bn.running_var.copy_(torch.rand(bn.running_var.shape, generator=g) + 0.5)
            bn.weight.copy_(1.0 + 0.1 * torch.randn(bn.weight.shape, generator=g))
            bn.bias.copy_(0.1 * torch.randn(bn.bias.shape, generator=g))


DUMP_BUDGET = 64 * 2 ** 20  # bytes --dump-outputs writes in all
DUMP_SAMPLE = 6 * 2 ** 20   # elements kept of a larger output (ctc_out: T x B x vocab logits)


def dump_outputs(out, dirname):
    """--dump-outputs: every tensor of ``out`` (the output mapping the timed path hands its caller), as
    DIR/<field>.npy (float32; lengths float64).  An output of more than DUMP_SAMPLE elements is written as
    DIR/<field>_sample.npy: its elements at DUMP_SAMPLE flat indices drawn with a fixed seed, in index order,
    so two builds given the same arguments can be compared element for element."""
    import numpy as np
    arrays = {}
    for name, t in out.items():
        if not isinstance(t, torch.Tensor) or name == "src_tokens":  # src_tokens is the input batch
            continue
        if t.numel() > DUMP_SAMPLE:
            g = torch.Generator().manual_seed(0)
            idx = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=g).sort().values
            t, name = t.reshape(-1)[idx.to(t.device)], name + "_sample"
        arrays[name] = t.to(torch.float64 if name == "src_lengths" else torch.float32).cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BUDGET:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte budget" % (total, DUMP_BUDGET))
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


# ------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index, interval_ms=20):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", str(int(interval_ms))], stdout=self.f,
                stderr=subprocess.DEVNULL) if interval_ms > 0 else None
        except OSError:
            self.p = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [s.strip() for s in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower() == "active":
                    reasons.add(n)
        os.unlink(self.f.name)
        if sm:
            out = dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons),
                       samples=len(sm))
        return out


# ------------------------------------------------------------------------------ per-kernel timing
class KernelProfile:
    """Wraps the op entry points with CUDA events (on the launching stream) to attribute device
    time and algorithmic work to kernel families."""

    def __init__(self, ops):
        self.ops, self.records, self.saved, self.post = ops, [], {}, False

    def _wrap(self, name, work):
        fn = getattr(self.ops, name)
        self.saved[name] = fn

        def wrapper(*a, **k):
            if name == "cmvn":
                self.post = False  # a new step starts: rows are the uncompressed ones again
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out = fn(*a, **k)
            e.record()
            # linear_ln is the same kernel family as linear (folded-LayerNorm epilogues)
            self.records.append(("linear" if name in ("linear_ln", "linear_argmax") else name, s, e,
                                 work(a, k, out)))
            if name == "ctc_compress":
                self.post = True  # later launches see only the compressed (valid) rows
            return out
        setattr(self.ops, name, wrapper)

    def __enter__(self):
        def valid_rows(M):
            return sum(self.new_lengths) if self.post else sum(self.att_lengths)

        def lin(a, k, out):
            M, K = a[0].shape
            M = valid_rows(M)
            N = a[1].shape[0]
            if isinstance(out, tuple):  # linear_ln producer side: (out, bf16 copy, row statistics)
                out = out[0]
                extra = M * N * 2 + M * ((N + 127) // 128) * 8
            else:
                extra = 0
            by = (M * K + N * K) * 2 + M * N * (4 if out.dtype == torch.float32 else 2) + extra
            if k.get("residual") is not None:
                by += M * N * 4
            # which kernel serves this launch (csrc/gemm2_tcgen05.cu, csrc/gemm_tcgen05.cu)
            if k.get("remap") is not None:
                sub = "gemm_bf16_kernel (fc3: row remap + pos-emb epilogue)"
            elif k.get("residual") is None and out.dtype == torch.float32:
                sub = "gemm2_kernel<f32 out> (fc3 + ReLU)"
            elif k.get("residual") is not None:
                sub = "gemm2_kernel<f32 out + residual (+ bf16 copy, LN statistics)> (out_proj, fc2)"
            else:
                sub = "gemm2_kernel<bf16 out> (qkv, fc1, ctc_fc)"
            return dict(flops=2.0 * M * N * K, bytes=by, sub=sub)

        def lin_am(a, k, out):  # ctc_fc with the fused arg-max epilogue: fp32 logits written once
            M, K = a[0].shape
            M = valid_rows(M)
            N = a[1].shape[0]
            return dict(flops=2.0 * M * N * K, bytes=(M * K + N * K) * 2 + M * N * 4 + M * ((N + 127) // 128) * 16,
                        sub="gemm2_kernel<f32 out + arg-max epilogue> (ctc_fc)")

        def att(a, k, out):
            qkv, lengths, L, B, H = a[:5]
            ln = self.new_lengths if self.post else self.att_lengths
            return dict(flops=sum(4.0 * n * n * 64 * H for n in ln),
                        bytes=sum(n * H * 64 * 2 * 4 for n in ln))

        def ln_(a, k, out):
            M, D = a[0].shape
            M = valid_rows(M)
            return dict(flops=0.0, bytes=M * D * (4 + out.element_size()))

        def argmax(a, k, out):
            lg, lengths, L, B, V = a[:5]
            return dict(flops=0.0, bytes=sum(self.att_lengths) * V * lg.element_size() + L * B * 8)

        def compress(a, k, out):
            x = a[0]
            return dict(flops=0.0, bytes=(sum(self.att_lengths) + sum(self.new_lengths)) * x.shape[-1] * 4)

        def conv1(a, k, out):
            return dict(flops=2.0 * out.numel() * 9, bytes=a[0].numel() * 4 + out.numel() * 2)

        def conv2(a, k, out):
            C = out.shape[-1]
            return dict(flops=2.0 * out.numel() * 9 * C, bytes=a[0].numel() * 2 + out.numel() * 2)

        def conv2p(a, k, out):
            C = out.shape[-1]
            return dict(flops=2.0 * out.numel() * 9 * C, bytes=a[0].numel() * 2 + out.numel() * 2)

        def cmvn(a, k, out):
            return dict(flops=0.0, bytes=a[0].numel() * 4 * 3)

        def other(a, k, out):
            return dict(flops=0.0, bytes=0)
        def stats(a, k, out):
            M, D = a[0].shape
            return dict(flops=0.0, bytes=valid_rows(M) * D * (4 + 2))

        def embed(a, k, out):  # read fp32 (+ table rows), write fp32 + bf16
            M, D = a[0].shape
            return dict(flops=0.0, bytes=M * D * (4 + 4 + 4 + 2))

        for name, w in [("linear", lin), ("linear_ln", lin), ("linear_argmax", lin_am), ("row_stats_cast", stats),
                        ("embed_remap_stats", embed), ("attention", att),
                        ("layernorm", ln_), ("ctc_argmax", argmax),
                        ("ctc_compress", compress), ("ctc_segment", other), ("conv1_relu_bn", conv1),
                        ("conv2_relu_bn", conv2), ("conv1_relu_bn_planes", conv1),
                        ("conv2_relu_bn_planes", conv2p), ("cmvn", cmvn), ("cast_bf16", other),
                        ("lengths_to_mask", other)]:
            self._wrap(name, w)
        return self

    def __exit__(self, *exc):
        for name, fn in self.saved.items():
            setattr(self.ops, name, fn)

    def summary(self, steps):
        torch.cuda.synchronize()
        agg = {}
        for name, s, e, w in self.records:
            for key in (name, w.get("sub")):
                if key is None:
                    continue
                d = agg.setdefault(key, dict(ms=0.0, flops=0.0, bytes=0.0, launches=0))
                d["ms"] += s.elapsed_time(e)
                d["flops"] += w["flops"]
                d["bytes"] += w["bytes"]
                d["launches"] += 1
        out = {}
        for name, d in agg.items():
            sec = d["ms"] * 1e-3
            out[name] = dict(ms_per_step=round(d["ms"] / steps, 4), launches_per_step=d["launches"] // steps,
                             tflops=round(d["flops"] / sec / 1e12, 2) if d["flops"] else None,
                             gbs=round(d["bytes"] / sec / 1e9, 1) if d["bytes"] else None)
        # algorithmic FLOPs of one step (every kernel family once; sub-families are views of `linear`)
        self.flops_per_step = sum(w["flops"] for _, _, _, w in self.records) / steps
        return out


# ------------------------------------------------------------------------------ our arm
def run_ours(args, rank, world, local_rank):
    from fbkst_b200 import ops
    from fbkst_b200.config import build_encoder
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    cfg = CONFIGS[args.config]
    model, lengths = cfg["model"], cfg["lengths"]
    B, T, Fd = len(lengths), max(lengths), model["feat_dim"]
    torch.manual_seed(0)
    enc = build_encoder(model, None, device="cpu")
    randomise_norm_stats(enc, 1)
    enc = enc.to(dev).eval()
    enc.use_cuda_graph = not args.no_graph  # one captured graph per input shape (see encoder._replay)
    L = ((T + 1) // 2 + 1) // 2
    plan = label_plan(L, B, model["vocab"], seed=7 + rank).to(dev)

    # run-structured logit injection (SURVEY F9): logits[t, b, plan[t, b]] += margin inside the ctc_fc epilogue
    # (same effect as a forward hook on ctc_fc -- which the tests use -- but keeps the fused arg-max epilogue)
    if model["ctc_layer"] > 0:
        if args.ctc_hook:
            enc.ctc_fc.register_forward_hook(lambda m, i, o: o.scatter_add(
                2, plan.unsqueeze(-1), torch.full_like(o[..., :1], CTC_MARGIN)))
        else:
            enc.ctc_logit_bump = (plan.to(torch.int32).contiguous(), CTC_MARGIN)

    n_batches = 9  # rotating inputs: 9 x 15.4 MB = 138 MB > the 126 MB L2 (cfg2)
    host = [make_batch(lengths, Fd, 1234 + rank * 100 + i) for i in range(n_batches)]
    host = [(x.pin_memory(), l) for x, l in host]
    dev_batches = [(x.to(dev), l) for x, l in host]
    len32 = torch.tensor(lengths, dtype=torch.int32, device=dev)
    frames = float(sum(lengths))
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step_resident(i):
        x, l = dev_batches[i % n_batches]
        xn = ops.cmvn(x, len32)
        return enc(xn, l)  # lengths stay on the host: no D2H sync for shape logic

    from fbkst_b200.pipeline import EncoderPipeline
    pipe = EncoderPipeline(enc, normalize=True, device=dev)

    def run_device(n):
        """n steps with the batches already in HBM, through the same compute lanes as the host-buffer
        API (CMVN + encoder forward per batch, `lanes` batches in flight)."""
        last = None
        for o in pipe.run_device(dev_batches[i % n_batches] for i in range(n)):
            last = o
        return last

    def run_e2e(n):
        """n steps through the public host-buffer API: pinned host batch -> H2D -> CMVN -> encoder
        -> D2H of encoder_out + lengths (copies overlap the kernels of the neighbouring steps)."""
        last = None
        stamps = [time.perf_counter()]
        for res, nl in pipe.run(host[i % n_batches] for i in range(n)):
            last = (res, nl)
            stamps.append(time.perf_counter())
        run_e2e.stamps = stamps  # [start, result 1, ..., result n]
        return last

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank, args.clock_interval_ms) if rank == 0 else None  # warm-up + timed regions
    for i in range(args.warmup):
        step_resident(i)
    run_device(max(args.warmup, 8))  # every lane's graph, every staging slot and pinned buffer exists
    run_e2e(max(args.warmup, 8))
    barrier()
    # the host is part of the e2e loop: keep CPython's cyclic collector (a full pass over torch's object
    # graph costs tens of ms) out of the timed regions; re-enabled before the attribution pass
    import gc
    gc.collect()
    gc.freeze()
    gc.disable()

    # ---- timed region 1: inputs resident in HBM, K steps back to back (throughput: `lanes` batches in
    # flight); rotating inputs larger than L2, and every step streams > 1 GB of activations through it
    launches0 = ops.LAUNCHES
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    ev0.record()
    out = run_device(args.steps)
    ev1.record()
    barrier()
    wall = time.perf_counter() - wall0
    launches = (ops.LAUNCHES - launches0) // args.steps
    dev_ms = ev0.elapsed_time(ev1)
    new_frames = float(out.src_lengths.sum().item())
    if args.dump_outputs and rank == 0:  # before any later launch reuses the graph buffers `out` aliases
        dump_outputs(out._asdict(), args.dump_outputs)

    # ---- informative: ONE forward at a time, L2 flushed (256 MB write, untimed) before each and ~1 ms of
    # untimed GPU-side delay so that the host enqueues the step while the GPU is still busy (no launch
    # latency inside the event pair): the cold-cache latency of a single batch
    evs = []
    for i in range(min(args.steps, 10)):
        flush.fill_(i & 0xFF)
        torch.cuda._sleep(LOOKAHEAD_CYCLES)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        step_resident(i)
        e.record()
        evs.append((s, e))
    barrier()
    step_ms = [s.elapsed_time(e) for s, e in evs]

    # ---- timed region 2: end to end from pinned host buffers (H2D + D2H inside); its own warm-up runs
    # right before it (the first host-buffer pass after a stretch of device-only work has been seen to
    # deliver its first result tens of ms late on a fresh box)
    run_e2e(max(args.warmup, 8))
    barrier()
    t0 = time.perf_counter()
    res, nl = run_e2e(args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    first_result_ms = (run_e2e.stamps[1] - run_e2e.stamps[0]) * 1e3
    gaps = [b - a for a, b in zip(run_e2e.stamps[1:], run_e2e.stamps[2:])] or [0.0]
    clocks = sampler.stop() if sampler else None

    t = torch.tensor([dev_ms, e2e_s * 1e3, max(gaps) * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    dev_ms, e2e_ms, worst_gap_ms = t.tolist()

    gc.enable()
    # ---- per-kernel attribution (separate, untimed pass; same stream, CUDA events)
    kern = None
    if rank == 0:
        enc.use_cuda_graph = False  # the attribution pass needs the individual launches
        with KernelProfile(ops) as kp:
            kp.att_lengths = [((n + 1) // 2 + 1) // 2 for n in lengths]
            kp.new_lengths = out.src_lengths.tolist()
            kp.L_pre = L
            prof_steps = 3
            step_resident(0)  # eager warm-up (allocations, workspaces) before the events
            torch.cuda.synchronize()
            kp.records.clear()
            # keep the GPU behind the CPU so that no launch gap leaks into an event interval
            torch.cuda._sleep(int(0.06 * 1.9e9))
            for i in range(prof_steps):
                step_resident(i)
            kern = kp.summary(prof_steps)
            flops_per_step = kp.flops_per_step
        enc.use_cuda_graph = not args.no_graph

    # ---- sustained figure: >= `--soak-seconds` of back-to-back steps (the B200 settles at its power
    # cap well below the 1965 MHz of a 45 ms burst); every rank runs it, rank 0 reports
    sustained = None
    if args.soak_seconds > 0:
        n_soak = max(args.steps, int(args.soak_seconds / (dev_ms / args.steps * 1e-3)))
        soak_sampler = ClockSampler(local_rank, 100) if rank == 0 else None
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        run_device(n_soak)
        s1.record()
        barrier()
        soak_ms = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device=dev)
        if world > 1:
            torch.distributed.all_reduce(soak_ms, op=torch.distributed.ReduceOp.MAX)
        soak_clk = soak_sampler.stop() if soak_sampler else None
        sustained = dict(steps=n_soak, seconds=round(soak_ms.item() * 1e-3, 3),
                         ms_per_step=round(soak_ms.item() / n_soak, 4),
                         value=round(world * frames * n_soak / (soak_ms.item() * 1e-3), 1),
                         unit="frames/s", clocks=soak_clk)

    if rank != 0:
        return None
    # parity sample: batch 0 through the timed code path (graph replay unless --no-graph), compared in
    # main() with the CPU arm's output for the same utterances, weights and label plan
    o0 = step_resident(0)
    torch.cuda.synchronize()
    n_par = min(8, B)
    parity_sample = dict(encoder_out=o0.encoder_out[:, :n_par].float().cpu(),
                         src_lengths=o0.src_lengths[:n_par].cpu().tolist(),
                         x=host[0][0][:n_par].clone(), lengths=lengths[:n_par], plan=plan[:, :n_par].cpu())
    pk = peaks()
    ms_per_step = dev_ms / args.steps
    value = world * frames / (ms_per_step * 1e-3)
    # Roofline of the dominant kernel = the tcgen05 linear kernel, ALL its instantiations together (qkv,
    # out_proj, fc1, fc2, fc3, ctc_fc: one source, three epilogues), not the best of them.  The
    # attribution pass is three eager steps (~10 ms at full clocks), so the denominator is the BURST peak;
    # the `sustained` block below relates the whole step to the sustained peak over a >= 2 s soak.
    kern_ms = sum(v["ms_per_step"] for k, v in kern.items() if not k.startswith("gemm"))
    lin = kern["linear"]

    def frac_of(k, peak):
        return round(kern[k]["tflops"] / peak, 4) if kern.get(k) and kern[k]["tflops"] else None
    tensor_kernels = {k: dict(tflops=kern[k]["tflops"], frac_of_burst=frac_of(k, pk["tf_burst"]),
                              ms_per_step=kern[k]["ms_per_step"],
                              share_of_step=round(kern[k]["ms_per_step"] / kern_ms, 4))
                      for k in kern if kern[k]["tflops"] and k != "conv1_relu_bn"}
    hbm_kernels = {k: dict(gbs=kern[k]["gbs"], frac_of_hbm=round(kern[k]["gbs"] / pk["hbm"], 4),
                           ms_per_step=kern[k]["ms_per_step"])
                   for k in ("cmvn", "conv1_relu_bn", "embed_remap_stats", "ctc_argmax", "ctc_compress",
                             "layernorm", "row_stats_cast") if kern.get(k) and kern[k]["gbs"]}
    roofline = dict(kernel="gemm2_kernel, all instantiations (qkv, out_proj, fc1, fc2, fc3, ctc_fc), "
                           "%d launches/step, %.1f%% of the step" % (
                               lin["launches_per_step"], 100 * lin["ms_per_step"] / kern_ms),
                    bound="tensor", achieved=lin["tflops"], peak=pk["tf_burst"], unit="TFLOP/s",
                    frac=round(lin["tflops"] / pk["tf_burst"], 4),
                    traffic=int(sum(NCU_TRAFFIC[k] * kern[k]["launches_per_step"] for k in NCU_TRAFFIC
                                    if k in kern) / max(1, sum(kern[k]["launches_per_step"]
                                                               for k in NCU_TRAFFIC if k in kern))),
                    traffic_unit="bytes/launch (dram read+write, ncu --set full, profiles/; mean over the "
                                 "family's launches)",
                    algorithmic="flops of the valid rows of every launch / CUDA-event time of the "
                                "launches (separate attribution pass of 3 eager steps, same stream)",
                    peak_source=pk["src"] + " (burst bf16: short attribution window at full clocks)",
                    tensor_kernels=tensor_kernels, hbm_kernels=hbm_kernels,
                    hbm_peak_gbs=pk["hbm"],
                    whole_step=dict(gflop_per_step=round(flops_per_step / 1e9, 1),
                                    mflop_per_frame=round(flops_per_step / frames / 1e6, 2),
                                    tflops=round(flops_per_step / (ms_per_step * 1e-3) / 1e12, 1),
                                    frac_of_burst=round(flops_per_step / (ms_per_step * 1e-3) / 1e12
                                                        / pk["tf_burst"], 4)),
                    sustained=sustained and dict(
                        sustained, tflops=round(flops_per_step * sustained["steps"] /
                                                (sustained["seconds"]) / 1e12, 1),
                        frac_of_sustained_peak=round(flops_per_step * sustained["steps"] /
                                                     sustained["seconds"] / 1e12 / pk["tf_sust"], 4),
                        peak=pk["tf_sust"]))
    h2d = host[0][0].numel() * 4
    d2h = res.numel() * res.element_size() + nl.numel() * nl.element_size()
    result = dict(
        metric="encoder fbank frames/sec", value=round(value, 1), unit="frames/s", n_gpus=world,
        steps=args.steps, warmup=args.warmup, ms_per_step=round(ms_per_step, 4),
        higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
        config=dict(workload=cfg["name"], per_gpu_batch="%dx%dx%d" % (B, T, Fd),
                    frames_per_step_per_gpu=frames, vocab=model["vocab"],
                    ctc_logit_injection="run-structured labels (geometric mean 3, 50%% blank), margin %g" % CTC_MARGIN,
                    compression_ratio=round(new_frames / sum(((n + 1) // 2 + 1) // 2 for n in lengths), 3),
                    cache="%d rotating input batches (%.0f MB in total vs the 126 MB L2) plus the activations "
                          "every step streams through L2 (> 1 GB at cfg2); no flush inside the timed region "
                          "(steps run back to back, %d in flight); single_forward_ms is the flushed, "
                          "one-at-a-time figure"
                          % (n_batches, n_batches * host[0][0].numel() * 4 / 1e6, pipe.lanes),
                    compute_lanes=pipe.lanes,
                    launch="eager" if args.no_graph else "CUDA graph replay of the encoder body",
                    parallelism="utterance-batch sharded x%d, no forward collective" % world),
        e2e=dict(value=round(world * frames / (e2e_ms * 1e-3 / args.steps), 1), unit="frames/s",
                 h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                 ms_per_step=round(e2e_ms / args.steps, 4),
                 api="fbkst_b200.pipeline.EncoderPipeline.run (pinned host batches in, pinned host "
                     "encoder_out + lengths out; wall clock over all steps incl. pipeline fill/drain)",
                 compute_lanes=pipe.lanes,
                 result_to_result_ms=dict(median=round(statistics.median(gaps) * 1e3, 3),
                                          max=round(max(gaps) * 1e3, 3), at_step=gaps.index(max(gaps)) + 1,
                                          max_over_ranks=round(worst_gap_ms, 3),
                                          first_result_ms=round(first_result_ms, 3),
                                          note="host clock between consecutive results (rank 0; max over "
                                               "ranks separately)")),
        gpu_launches=launches, clocks=clocks, roofline=roofline, kernels=kern,
        wall_ms_per_step=round(wall * 1e3 / args.steps, 4), impl="ours",
        single_forward_ms=dict(min=round(min(step_ms), 4), median=round(statistics.median(step_ms), 4),
                               max=round(max(step_ms), 4),
                               note="rank 0: one forward at a time, L2 flushed (256 MB write) before each, "
                                    "CUDA events per step; not the throughput figure"))
    return result, enc, parity_sample



# ------------------------------------------------------------------------------ cfg4: training step
def _reference_root():
    env = os.environ.get("FBKST_REFERENCE_ROOT")
    if env:
        return env
    for cand in ("/root/reference", os.path.join(ROOT, "baseline", "_ref")):
        if os.path.isdir(os.path.join(cand, "examples", "speech_recognition")):
            return cand
    return None


def run_train(args, rank, world, local_rank):
    """BASELINE configs[3]: one optimisation step of the ST model the way fairseq's trainer runs it
    (fairseq/trainer.py:335-443 -> tasks/speech_recognition.py:234-263): criterion(model, sample) with the
    plugin's model (`--arch conv_transformer_big2_b200`: OUR encoder forward + backward kernels, fairseq's own
    TransformerDecoder under bf16 autocast) and criterion (`ctc_multi_loss_b200`: CTC loss on our kernels +
    fairseq's label-smoothed CE), loss.backward(), the reference's own LegacyDistributedDataParallel
    (`--ddp-backend no_c10d`, README.md:142: ONE flat NCCL all-reduce after the backward), Adam step.
    Everything outside the encoder / CTC loss is the reference's code, imported from baseline/_ref."""
    root = _reference_root()
    if root is None:
        raise RuntimeError("cfg4 needs the reference package (baseline/_ref; run baseline/make_ref.py)")
    plugin = os.path.join(ROOT, "fbk-fairseq-st_b200", "fbkst_b200", "plugin")
    sys.path.insert(0, plugin)
    import compat
    compat.apply_numpy()
    sys.path.insert(0, root)
    import warnings
    warnings.simplefilter("ignore")
    from fairseq import criterions, options, utils
    utils.import_user_module(argparse.Namespace(user_dir=plugin))
    from fairseq.data import Dictionary
    from fairseq.models import MODEL_REGISTRY
    from fbkst_b200 import ops

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    cfg = CONFIGS[args.config]
    model_cfg, dec, lengths = cfg["model"], cfg["decoder"], cfg["lengths"]
    B, T, Fd = len(lengths), max(lengths), model_cfg["feat_dim"]

    def make_dict(n, blank):
        d = Dictionary()
        for i in range(n - len(d) - (1 if blank else 0)):
            d.add_symbol("w%d" % i)
        if blank:
            d.add_symbol("<ctc_blank>")
        return d

    class Task:
        source_dictionary = make_dict(model_cfg["vocab"], True)
        target_dictionary = make_dict(dec["tgt_vocab"], False)

        def build_criterion(self, a):
            return criterions.build_criterion(a, self)
    task = Task()
    parser = options.get_training_parser()
    fa = options.parse_args_and_arch(parser, [
        "/tmp/nodata", "--user-dir", plugin, "--arch", "conv_transformer_big2_b200",
        "--task", "speech_translation_with_transcription", "--criterion", "ctc_multi_loss_b200",
        "--underlying-criterion", "label_smoothed_cross_entropy", "--label-smoothing", "0.1",
        "--ctc-encoder-layer", str(model_cfg["ctc_layer"]), "--ctc-compress-out",
        "--ctc-compress-strategy", model_cfg["ctc_strategy"], "--no-attn-2d", "--distance-penalty", "log",
        "--input-feat-per-channel", str(Fd), "--encoder-layers", str(model_cfg["layers"]),
        "--encoder-embed-dim", str(model_cfg["embed_dim"]), "--encoder-ffn-embed-dim", str(model_cfg["ffn_dim"]),
        "--encoder-attention-heads", str(model_cfg["heads"]), "--decoder-layers", str(dec["layers"]),
        "--max-tokens", "12000", "--skip-normalization", "--dropout", "0.1", "--ddp-backend", "no_c10d"])
    torch.manual_seed(0)
    model = MODEL_REGISTRY["conv_transformer_b200"].build_model(fa, task).to(dev)
    criterion = criterions.build_criterion(fa, task).to(dev)
    model.train()
    criterion.train()
    n_params = sum(p.numel() for p in model.parameters())
    n_enc = sum(p.numel() for p in model.encoder.parameters())
    ddp = model
    if world > 1:
        from fairseq.legacy_distributed_data_parallel import LegacyDistributedDataParallel
        ddp = LegacyDistributedDataParallel(model, world, process_group=None, buffer_size=2 ** 28)
        for name in ("encoder", "decoder", "get_normalized_probs", "get_targets", "max_positions"):
            setattr(ddp, name, getattr(model, name))  # what DistributedFairseqModel forwards
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, betas=(0.9, 0.98), fused=True)

    L = ((T + 1) // 2 + 1) // 2
    plan = label_plan(L, B, model_cfg["vocab"], seed=7 + rank).to(dev)
    if args.ctc_hook:  # the injection as an nn.Module forward hook (out of place: one extra copy of the logits)
        model.encoder.ctc_fc.register_forward_hook(
            lambda m, i, o: o.scatter_add(2, plan.unsqueeze(-1), torch.full_like(o[..., :1], CTC_MARGIN)))
    else:  # the encoder's built-in injection, as in the forward benchmark
        model.encoder.ctc_logit_bump = (plan.to(torch.int32).contiguous(), CTC_MARGIN)
    g = torch.Generator().manual_seed(99 + rank)
    n_batches = 4
    samples = []
    for i in range(n_batches):
        x, l = make_batch(lengths, Fd, 1234 + rank * 100 + i)
        U, U1 = dec["tgt_len"], dec["transcript_len"]
        tgt = torch.randint(4, dec["tgt_vocab"] - 1, (B, U), generator=g)
        tgt[:, -1] = task.target_dictionary.eos()
        prev = torch.cat([torch.full((B, 1), task.target_dictionary.eos()), tgt[:, :-1]], 1)
        tr = torch.randint(4, model_cfg["vocab"] - 2, (B, U1), generator=g)
        trl = torch.full((B,), U1, dtype=torch.long)
        samples.append(utils.move_to_cuda(dict(
            net_input=dict(src_tokens=x, src_lengths=l, prev_output_tokens=prev), target=tgt,
            transcript_target=tr, transcript_target_lengths=trl, ntokens=B * U, nsentences=B)))
    frames = float(sum(lengths))

    marks = {}

    def step(i, timed=None):
        s = samples[i % n_batches]
        ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
        e = [ev() for _ in range(5)] if timed is not None else None
        torch.manual_seed(1000 + i)  # dropout seed source (fairseq: trainer.py:655-661)
        opt.zero_grad(set_to_none=True)
        if e:
            e[0].record()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss, sample_size, log = criterion(ddp, s)
        if e:
            e[1].record()
        loss.backward()  # the legacy DDP all-reduce fires at the end of the backward (one flat buffer)
        if e:
            e[2].record()
        opt.step()
        if e:
            e[3].record()
            timed.append(e)
        return loss

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank, args.clock_interval_ms) if rank == 0 else None
    for i in range(max(args.warmup, 3)):
        step(i)
    barrier()
    if os.environ.get("FBKST_TRAIN_PROFILE") and rank == 0:  # informative per-kernel table on stderr (untimed)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(2):
                step(i)
            torch.cuda.synchronize()
        rows = sorted(((getattr(e, "device_time_total", 0), e.count, e.key) for e in prof.key_averages()), reverse=True)
        tot = sum(r[0] for r in rows if not r[2].startswith("Optimizer.step"))
        sys.stderr.write("per-kernel device time over 2 training steps: %.2f ms/step\n" % (tot / 2e3))
        for t, n, k in rows[:60]:
            sys.stderr.write("%8.3f ms/step %5.1f%%  n=%-4d %s\n" % (t / 2e3, 100 * t / max(tot, 1), n // 2, k[:120]))
    if os.environ.get("FBKST_TRAIN_CPROFILE") and rank == 0:  # informative host-side profile (untimed)
        import cProfile
        import io
        import pstats
        pr = cProfile.Profile()
        pr.enable()
        for i in range(3):
            step(i)
        torch.cuda.synchronize()
        pr.disable()
        for key in ("tottime", "cumulative"):
            buf = io.StringIO()
            pstats.Stats(pr, stream=buf).sort_stats(key).print_stats(45)
            sys.stderr.write("host profile of 3 training steps, by %s\n%s\n" % (key, buf.getvalue()))
    launches0 = ops.LAUNCHES
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(args.steps):
        last = step(i)
    ev1.record()
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(dict(loss=last.detach()), args.dump_outputs)
    launches = (ops.LAUNCHES - launches0) // args.steps
    # e2e: batches start in pinned HOST memory (H2D inside), the loss is read back on the host every step
    host = [utils.apply_to_sample(lambda t: t.cpu().pin_memory(), s) for s in samples]
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        samples[i % n_batches] = utils.apply_to_sample(lambda t: t.to(dev, non_blocking=True), host[i % n_batches])
        lv = step(i).item()
    barrier()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop() if sampler else None
    # attribution (untimed region): forward / backward(+all-reduce) / optimizer split with CUDA events
    timed = []
    for i in range(3):
        step(i, timed)
    torch.cuda.synchronize()
    split = dict(forward_and_loss_ms=round(sum(e[0].elapsed_time(e[1]) for e in timed) / 3, 3),
                 backward_and_allreduce_ms=round(sum(e[1].elapsed_time(e[2]) for e in timed) / 3, 3),
                 optimizer_ms=round(sum(e[2].elapsed_time(e[3]) for e in timed) / 3, 3))
    # the all-reduce alone: the same flat buffer the legacy wrapper uses (fp32, all parameters)
    ar_ms = None
    if world > 1:
        buf = torch.empty(n_params, dtype=torch.float32, device=dev)
        torch.distributed.all_reduce(buf)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(5):
            torch.distributed.all_reduce(buf)
        a1.record()
        torch.cuda.synchronize()
        ar_ms = a0.elapsed_time(a1) / 5
    t = torch.tensor([dev_ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    dev_ms, e2e_ms = t.tolist()
    if rank != 0:
        return None
    ms_per_step = dev_ms / args.steps
    h2d = sum(v.numel() * v.element_size() for v in
              [host[0]["net_input"]["src_tokens"], host[0]["net_input"]["src_lengths"],
               host[0]["net_input"]["prev_output_tokens"], host[0]["target"], host[0]["transcript_target"],
               host[0]["transcript_target_lengths"]])
    return dict(
        metric="encoder fbank frames/sec", value=round(world * frames / (ms_per_step * 1e-3), 1), unit="frames/s",
        n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=round(ms_per_step, 4),
        higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
        config=dict(workload=cfg["name"], per_gpu_batch="%dx%dx%d" % (B, T, Fd),
                    frames_per_step_per_gpu=frames, parameters=n_params, encoder_parameters=n_enc,
                    step="criterion(model, sample) [fairseq ctc_multi_loss_b200] -> backward -> flat gradient "
                         "all-reduce (fairseq LegacyDistributedDataParallel, no_c10d) -> Adam",
                    encoder="fbkst_b200 forward + backward kernels (train mode: BatchNorm batch statistics, "
                            "dropout 0.1 / conv 0.1 / attention 0.1 / relu 0.1)",
                    decoder="fairseq TransformerDecoder (PyTorch, bf16 autocast), label-smoothed CE",
                    cache="%d rotating batches; every step streams several GB of saved activations" % n_batches,
                    parallelism="data parallel x%d, one flat NCCL all-reduce per step" % world),
        e2e=dict(value=round(world * frames / (e2e_ms * 1e-3 / args.steps), 1), unit="frames/s",
                 h2d_bytes_per_step=h2d, d2h_bytes_per_step=4, ms_per_step=round(e2e_ms / args.steps, 4),
                 api="fairseq criterion(model, sample) on the plugin model; pinned host sample in, loss.item() out"),
        gpu_launches=launches, clocks=clocks, impl="ours", train_step_split=split,
        allreduce=dict(ms=None if ar_ms is None else round(ar_ms, 3), bytes=n_params * 4,
                       share_of_step=None if ar_ms is None else round(ar_ms / ms_per_step, 4),
                       note="flat fp32 gradient buffer, torch.distributed NCCL all_reduce timed alone (5 reps)"),
        final_loss=round(float(lv), 3),
        roofline=None, cpu_baseline=None)



# ------------------------------------------------------------------------------ cfg3: ragged, length-bucketed
def run_ragged(args, rank, world, local_rank):
    """BASELINE configs[2]: the cfg2 model with weighted / softmax pooling on RAGGED utterances (200..3000
    frames), partitioned across the ranks by length-bucketed batch (fbkst_b200.sharding: sort by length, cut
    into batches of <= 96 k padded frames with T quantised to 128 frames, deal every `world` consecutive
    -- near-equal-cost -- batches to the ranks of one step).  Every rank runs DIFFERENT batches with different
    shapes; no collective on the data path.  Weak scaling: the utterance pool grows with `world` so that every
    rank runs `--steps` batches.  Reported: aggregate valid frames/s over the slowest rank's device time, the
    per-rank time spread and the partition's padded-frame imbalance."""
    import random
    from fbkst_b200 import ops, sharding
    from fbkst_b200.config import build_encoder
    from fbkst_b200.pipeline import EncoderPipeline
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    cfg = CONFIGS["cfg3"]
    model = dict(cfg["model"], ctc_strategy=args.ctc_strategy or cfg["model"]["ctc_strategy"])
    Fd, PAD, MAXF = model["feat_dim"], 128, 96000
    rng = random.Random(20210421)  # the same pool on every rank
    pool = []
    want = world * args.steps
    pool_for = max(world, 8) * args.steps  # the SAME pool at every world size <= 8: the length mix per rank
    while True:                            # does not depend on N (weak scaling compares like with like)
        pool += [rng.randint(200, 3000) for _ in range(512)]
        batches = sharding.bucket_by_length(pool, MAXF, pad_multiple=PAD)
        if len(batches) >= pool_for + 1:  # + 1: the last (shortest, partly filled) batch is dropped
            break
    # `want` batches spread over the whole length range (every k-th of the sorted batch list)
    stride = (len(batches) - 1) // want
    batches = [batches[i * stride] for i in range(want)] if stride >= 1 else batches[:want]
    steps = sharding.shard_steps(batches, world)
    imbalance = sharding.step_imbalance(pool, steps, PAD)
    mine = [st[rank] for st in steps]

    torch.manual_seed(0)
    enc = build_encoder(model, None, device="cpu")
    randomise_norm_stats(enc, 1)
    enc = enc.to(dev).eval()
    enc.use_cuda_graph = not args.no_graph
    enc.max_graphs = 96
    Lmax, Bmax = (3072 + 3) // 4, MAXF // 256
    plan_big = label_plan(Lmax, Bmax, model["vocab"], seed=7).to(dev)
    plans = {}

    def plan_for(Lb, Bb):
        if (Lb, Bb) not in plans:
            plans[(Lb, Bb)] = plan_big[:Lb, :Bb].to(torch.int32).contiguous()
        return plans[(Lb, Bb)]
    enc.ctc_logit_bump = (plan_for, CTC_MARGIN)
    g = torch.Generator().manual_seed(1234 + rank)
    noise = torch.randn(MAXF + 3072, Fd, generator=g) * 3.0 + 1.0
    dev_batches, frames, padded = [], 0.0, 0.0
    for b in mine:
        lens = [pool[i] for i in b]
        T = sharding.padded_length(max(lens), PAD)
        x = torch.zeros(len(b), T, Fd)
        o = 0
        for k, n in enumerate(lens):
            x[k, :n] = noise[o:o + n]
            o = (o + n) % 3000
        dev_batches.append((x.to(dev), torch.tensor(lens, dtype=torch.long)))
        frames += sum(lens)
        padded += len(b) * T
    shapes = sorted({tuple(x.shape[:2]) for x, _ in dev_batches})
    pipe = EncoderPipeline(enc, normalize=True, device=dev)

    def run(n_rep):
        last = None
        for _ in range(n_rep):
            for o in pipe.run_device(iter(dev_batches)):
                last = o
        return last

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank, args.clock_interval_ms) if rank == 0 else None
    run(2)  # every shape's graph on both lanes exists (untimed)
    barrier()
    import gc
    gc.collect()
    gc.freeze()
    gc.disable()
    launches0 = ops.LAUNCHES
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    out = run(1)
    ev1.record()
    barrier()
    if args.dump_outputs and rank == 0:  # before the next pass reuses the graph buffers `out` aliases
        dump_outputs(out._asdict(), args.dump_outputs)
    gc.enable()
    my_ms = ev0.elapsed_time(ev1)
    # untimed: every output of one more pass over the rank's batches must be finite (a ragged stream in persistent
    # workspaces is where stale rows beyond a device-side limit would show: DESIGN.md 4e)
    bad = torch.zeros((), dtype=torch.int64, device=dev)
    for o in pipe.run_device(iter(dev_batches)):
        bad += (~torch.isfinite(o.encoder_out)).sum()
    last_lens = dev_batches[-1][1].tolist()
    ratio_last = float(out.src_lengths.sum().item()) / sum(((n + 1) // 2 + 1) // 2 for n in last_lens)
    launches = (ops.LAUNCHES - launches0) // max(1, len(dev_batches))
    clocks = sampler.stop() if sampler else None
    stats = torch.tensor([my_ms, frames, padded, float(bad.item())], dtype=torch.float64, device=dev)
    allr = [torch.zeros_like(stats) for _ in range(world)]
    if world > 1:
        torch.distributed.all_gather(allr, stats)
    else:
        allr = [stats]
    if rank != 0:
        return None
    ms = [float(t[0]) for t in allr]
    tot_frames = sum(float(t[1]) for t in allr)
    tot_padded = sum(float(t[2]) for t in allr)
    worst = max(ms)
    return dict(
        metric="encoder fbank frames/sec", value=round(tot_frames / (worst * 1e-3), 1), unit="frames/s",
        n_gpus=world, steps=len(mine), warmup=2 * len(mine), ms_per_step=round(worst / len(mine), 4),
        higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
        config=dict(workload="cfg2 model, ctc-compress %s @8, RAGGED utterances 200..3000 frames, length-bucketed "
                             "batches of <= 96 k padded frames (T quantised to 128), different batches per rank"
                             % model["ctc_strategy"],
                    utterances_in_pool=len(pool), steps_per_rank=len(mine), distinct_shapes_rank0=len(shapes),
                    shapes_rank0=["%dx%d" % s for s in shapes[:4]] + ["..."] + ["%dx%d" % s for s in shapes[-2:]],
                    valid_frames_total=tot_frames, padded_frames_total=tot_padded,
                    padding_overhead=round(tot_padded / tot_frames - 1.0, 4),
                    compression_ratio_last_batch_rank0=round(ratio_last, 3),
                    launch="eager" if args.no_graph else "CUDA graph replay, one graph per (shape, lane)",
                    parallelism="utterance-batch sharded x%d by fbkst_b200.sharding, no forward collective" % world,
                    cache="every batch is a different tensor (%.0f MB per rank in total)" % (padded * Fd * 4 / 1e6 / world)),
        rank_time_ms=dict(min=round(min(ms), 3), max=round(worst, 3), mean=round(sum(ms) / len(ms), 3),
                          spread=round(worst / min(ms), 4), per_rank=[round(m, 3) for m in ms]),
        nonfinite_outputs=int(sum(float(t[3]) for t in allr)),
        step_imbalance_padded_frames=round(imbalance, 4),
        e2e=None, gpu_launches=launches, clocks=clocks, impl="ours", roofline=None, cpu_baseline=None)


# ------------------------------------------------------------------------------ CPU baseline
def parity_numbers(ours, ref, lengths):
    """Both readings of the north_star's 2e-2 (bf16) over the valid positions of T x B x D outputs:
    max|a-b|/max|ref| and max over elements of |a-b| / (|ref| + rms(ref)), per utterance, worst case."""
    worst_max = worst_el = 0.0
    bad_ours = bad_ref = 0
    for b, n in enumerate(lengths):
        a, r = ours[:n, b].double(), ref[:n, b].double()
        d = (a - r).abs()
        if not bool(torch.isfinite(d).all()):  # (max() would silently drop a NaN)
            worst_max = worst_el = float("inf")
            bad_ours += int((~torch.isfinite(a)).sum())
            bad_ref += int((~torch.isfinite(r)).sum())
            continue
        worst_max = max(worst_max, (d.max() / r.abs().max().clamp_min(1e-12)).item())
        worst_el = max(worst_el, (d / (r.abs() + r.pow(2).mean().sqrt().clamp_min(1e-12))).max().item())
    return dict(max_rel=round(worst_max, 5), elementwise=round(worst_el, 5), tolerance=2e-2,
                utterances=len(lengths), nonfinite_ours=bad_ours, nonfinite_reference=bad_ref,
                criteria="max_rel = max|a-b|/max|ref|; elementwise = max(|a-b|/(|ref|+rms(ref))); both per "
                         "utterance over valid positions, worst utterance; lengths compared exactly")


def _container_state_dict(model):
    """The GPU arm's weights without a GPU: our encoder class is only a parameter container here
    (same constructor RNG stream as run_ours: torch.manual_seed(0), then randomise_norm_stats)."""
    from fbkst_b200.config import build_encoder
    torch.manual_seed(0)
    enc = build_encoder(model, None, device="cpu")
    randomise_norm_stats(enc, 1)
    return {k: v.detach().clone() for k, v in enc.state_dict().items()}


def cpu_reference(args, enc_state=None, steps=3, warmup=1, sample_utts=8, sample=None, budget_s=None):
    """The reference's CPU path on the host cores for a bounded sample of the workload (the first
    `sample_utts` utterances of the step; the padded extent stays the full batch's, SURVEY F5).

    kind "reference": the UNMODIFIED reference module (``ConvolutionalTransformerEncoder.forward``,
    conv_transformer.py:195-276, preceded by the dataset's ``apply_mv_norm``, data/data_utils.py:17-24)
    imported from /root/reference or its copy baseline/_ref (baseline/make_ref.py), eval mode, no grad,
    fp32, all host threads, loaded with the GPU arm's weights (strict state_dict).
    kind "port": the CPU oracle restatement, when no reference tree is present.
    With ``sample`` (the first utterances of the GPU arm's batch 0 and their label plan) the output is
    also returned for the bench line's `parity` key.  ``budget_s``: stop timing after that many seconds
    (at least one timed step)."""
    from oracle import encoder_oracle as O
    from oracle import ref_loader as R
    cfg = CONFIGS[args.config]
    model, lengths = cfg["model"], cfg["lengths"][:sample_utts]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = enc_state if enc_state is not None else _container_state_dict(model)
    sd = {k: v.detach().float().cpu() if v.is_floating_point() else v.detach().cpu() for k, v in sd.items()}
    T = max(cfg["lengths"])
    L = ((T + 1) // 2 + 1) // 2
    if sample is not None:
        x, l, plan = sample["x"], torch.tensor(sample["lengths"], dtype=torch.long), sample["plan"]
    else:
        x, l = make_batch(lengths, model["feat_dim"], 1234)
        if x.shape[1] < T:  # same padded extent as the full batch (SURVEY F5)
            x = torch.nn.functional.pad(x, (0, 0, 0, T - x.shape[1]))
        plan = label_plan(L, len(cfg["lengths"]), model["vocab"], seed=7)[:, :len(lengths)]
    hook = O.bump_hook(plan, CTC_MARGIN)

    ref_enc = None
    if R.available() and not args.port_baseline:
        ref_enc = R.build_reference_encoder(model, seed=0, randomize_bn=False)
        ref_enc.load_state_dict(sd, strict=True)
        ref_enc.eval()
        if model["ctc_layer"]:
            ref_enc.ctc_fc.register_forward_hook(lambda m, i, o: hook(o))
        from examples.speech_recognition.data.data_utils import apply_mv_norm

    def step():
        with torch.no_grad():
            xn = torch.zeros_like(x)
            if ref_enc is not None:
                for b, n in enumerate(lengths):  # data/fbank_dataset.py:44-45: per utterance
                    xn[b, :n] = apply_mv_norm(x[b, :n])
                o = R.run_reference_encoder(ref_enc, xn, l)
                return dict(encoder_out=o.encoder_out, src_lengths=o.src_lengths,
                            encoder_padding_mask=o.encoder_padding_mask)
            for b, n in enumerate(lengths):
                xn[b, :n] = O.cmvn(x[b, :n])
            return O.encoder_forward(sd, model, xn, l, ctc_logits_hook=hook if model["ctc_layer"] else None)
    t_start = time.perf_counter()
    for _ in range(warmup):
        ref = step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        ref = step()
        times.append(time.perf_counter() - t0)
        if budget_s is not None and time.perf_counter() - t_start > budget_s:
            break
    sec = statistics.median(times)
    cb = dict(value=round(sum(lengths) / sec, 1), unit="frames/s", cores=cores,
              kind="reference" if ref_enc is not None else "port",
              source=(R.REFERENCE_ROOT + " (unmodified ConvolutionalTransformerEncoder.forward + apply_mv_norm)")
              if ref_enc is not None else "oracle/encoder_oracle.py (CPU restatement)",
              sample="first %d of %d utterances of the step (%d frames), fp32, median of %d after %d warm-up"
                     % (len(lengths), len(cfg["lengths"]), sum(lengths), len(times), warmup),
              ms_per_sample=round(sec * 1e3, 2))
    return cb, ref


def reference_gpu_eager(args, enc_state, plan, steps=3):
    """Informative: the UNMODIFIED reference module in PyTorch eager on the same B200 (fp32, torch's
    default matmul/conv precision flags), same weights / batch / label plan.  This is what a user of the
    reference gets on this GPU today; not part of any ratio."""
    from oracle import ref_loader as R
    if not R.available() or not torch.cuda.is_available():
        return None
    cfg = CONFIGS[args.config]
    model, lengths = cfg["model"], cfg["lengths"]
    dev = torch.device("cuda", 0)
    try:
        ref = R.build_reference_encoder(model, seed=0, randomize_bn=False)
        ref.load_state_dict({k: v.detach().cpu() for k, v in enc_state.items()}, strict=True)
        ref = ref.to(dev).eval()
        pl = plan.to(dev)
        if model["ctc_layer"]:
            ref.ctc_fc.register_forward_hook(
                lambda m, i, o: o.scatter_add(2, pl.unsqueeze(-1), torch.full_like(o[..., :1], CTC_MARGIN)))
        from examples.speech_recognition.data.data_utils import apply_mv_norm
        x, l = make_batch(lengths, model["feat_dim"], 1234)
        x, l = x.to(dev), l.to(dev)

        def step():
            with torch.no_grad():
                xn = torch.zeros_like(x)
                for b, n in enumerate(lengths):
                    xn[b, :n] = apply_mv_norm(x[b, :n])
                return ref(xn, l)
        step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
        sec = (time.perf_counter() - t0) / steps
        return dict(value=round(sum(lengths) / sec, 1), unit="frames/s", ms_per_step=round(sec * 1e3, 2),
                    dtype="f32", steps=steps, source=R.REFERENCE_ROOT,
                    note="unmodified reference module, PyTorch eager on cuda:0 (cuDNN/cuBLAS), wall clock "
                         "incl. its per-utterance host syncs; informative only")
    except Exception as e:  # the old code base may not run on every torch build: report, do not fail
        return dict(unavailable="%s: %s" % (type(e).__name__, str(e)[:200]))


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU implementation of the path (see cpu_reference) on ALL the
    utterances of the step -- the same config / metric / unit as our arm; under torchrun rank 0 alone
    runs it.  It times --steps steps; --reference-budget-s stops it earlier (said in `cpu_baseline.sample`)."""
    if rank != 0:
        return None
    cfg = CONFIGS[args.config]
    cb, ref = cpu_reference(args, steps=max(1, args.steps), warmup=max(1, min(args.warmup, 2)),
                            sample_utts=len(cfg["lengths"]), budget_s=args.reference_budget_s)
    if args.dump_outputs:
        dump_outputs(ref, args.dump_outputs)
    return dict(metric="encoder fbank frames/sec", value=cb["value"], unit="frames/s", n_gpus=world,
                steps=args.steps, warmup=args.warmup, ms_per_step=cb["ms_per_sample"],
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                config=dict(workload=cfg["name"],
                            note="reference CPU path on the host cores: " + cb["source"]),
                impl="reference", cpu_baseline=cb,
                e2e=dict(value=cb["value"], unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))


def main():
    # A run that is still going after 25 minutes is stuck (the default line takes ~1 minute, the reference arm
    # a few seconds per step): dump every thread's Python stack and exit non-zero instead of hanging without a trace.
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("FBKST_BENCH_DEADLINE_S", "1500")), exit=True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS) + ["cfg3r"],
                    help="cfg2: headline; cfg3: one ragged bucket; cfg3r: ragged, length-bucketed, different batches "
                         "per rank (BASELINE configs[2]); cfg4: training step; cfg5: long-form")
    ap.add_argument("--ctc-strategy", default=None, choices=["avg", "weighted", "softmax"],
                    help="cfg3r: pooling strategy (default weighted)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--clock-interval-ms", type=int, default=20,
                    help="nvidia-smi sampling period for the `clocks` key (0 = no sampler)")
    ap.add_argument("--no-graph", action="store_true", help="launch kernel by kernel instead of graph replay")
    ap.add_argument("--ctc-hook", action="store_true",
                    help="inject the CTC label plan through a forward hook on ctc_fc (unfused logits + arg-max "
                         "kernels) instead of the fused epilogue's built-in bump")
    ap.add_argument("--port-baseline", action="store_true",
                    help="time the CPU oracle port even when the reference tree (baseline/_ref) is present")
    ap.add_argument("--reference-budget-s", type=float, default=None,
                    help="--impl reference: stop timing after this many seconds (>= 1 timed step; default: "
                         "time all --steps steps)")
    ap.add_argument("--soak-seconds", type=float, default=2.0,
                    help="length of the sustained-throughput soak reported under roofline.sustained (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (the encoder output tuple with a seeded "
                         "sample of ctc_out; cfg4: the loss) to DIR/<name>.npy, rank 0; inputs are seeded, so "
                         "runs with the same arguments can be compared")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # Only the JSON line may reach stdout: libraries (NCCL prints its version banner there) write
    # to fd 1 behind Python's back, so fd 1 is pointed at stderr for the whole run.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    if args.impl == "reference":
        r = run_reference(args, rank, world)
        if r is not None:
            emit(r)
        return
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.config in ("cfg4", "cfg3r"):
        r = (run_train if args.config == "cfg4" else run_ragged)(args, rank, world, local_rank)
        if rank == 0:
            emit(r)
        if world > 1:
            torch.distributed.barrier()
            torch.distributed.destroy_process_group()
        return
    r = run_ours(args, rank, world, local_rank)
    if rank == 0:
        result, enc, sample = r
        if not args.no_cpu_baseline and world == 1:  # reported on rank 0 at N=1 only
            sd = {k: v for k, v in enc.state_dict().items()}
            result["cpu_baseline"], ref = cpu_reference(args, enc_state=sd, sample=sample)
            # parity of the timed configuration itself: the GPU arm's batch 0 vs the CPU arm on the same
            # utterances / weights / label plan (lengths exact, floats under both 2e-2 criteria)
            nl = ref["src_lengths"].tolist()
            par = parity_numbers(sample["encoder_out"], ref["encoder_out"], nl)
            par["lengths_equal"] = nl == sample["src_lengths"]
            par["against"] = result["cpu_baseline"]["kind"] + " (" + result["cpu_baseline"]["source"] + ")"
            result["parity"] = par
            full_plan = label_plan(sample["plan"].shape[0], len(CONFIGS[args.config]["lengths"]),
                                   CONFIGS[args.config]["model"]["vocab"], seed=7)
            result["reference_gpu_eager"] = reference_gpu_eager(args, sd, full_plan)
        emit(result)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
