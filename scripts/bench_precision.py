"""bf16 against fp32 (split-TF32) encoder precision on the bench's workloads, in one process.

For cfg1 and cfg2 (bench.py's seeded inputs, weights and CTC label plan, CUDA-graph mode as the bench runs
it) the two precisions are timed alternately with CUDA events after warm-up.  Reported per config: frames/s
of each precision, both parity readings of each against the fp32 CPU oracle (first utterances of the batch),
and, when the reference package is present, the reference module in fp32 PyTorch eager on the same GPU.
Also the algorithmic rate of the split-TF32 GEMM alone (2 M N K per call, the 3 tensor passes not counted)
at the cfg2 fc1 shape, and the card name and power limit (read-only nvidia-smi query).

    python scripts/bench_precision.py [--configs cfg1,cfg2] [--steps 20] [--out profiles/x.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "fbk-fairseq-st_b200")]
import bench  # noqa: E402
from helpers import parity_report  # noqa: E402
from oracle import encoder_oracle as O  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "unavailable: %s" % e
    return dict(nvidia_smi=q, torch_name=torch.cuda.get_device_name(0))


def time_events(fn, steps):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / steps


def gemm_rate(steps):
    from fbkst_b200 import ops
    M, N, K = 64 * 375, 2048, 512  # cfg2 fc1
    a = torch.randn(M, K, device="cuda")
    w = torch.randn(N, K, device="cuda")
    out = torch.empty(M, N, device="cuda")
    for _ in range(3):
        ops.linear_f32(a, w, out=out)
    sec = time_events(lambda: ops.linear_f32(a, w, out=out), steps * 10)
    return dict(shape="M=%d N=%d K=%d" % (M, N, K), us=round(sec * 1e6, 1),
                algorithmic_tflops=round(2.0 * M * N * K / sec / 1e12, 1))


def run_config(name, steps, warmup, n_ref):
    from fbkst_b200 import ops
    from fbkst_b200.config import build_encoder
    cfg = bench.CONFIGS[name]
    model, lengths = cfg["model"], cfg["lengths"]
    B, T = len(lengths), max(lengths)
    L = ((T + 1) // 2 + 1) // 2
    torch.manual_seed(0)
    enc = build_encoder(model, None, device="cpu")
    bench.randomise_norm_stats(enc, 1)
    enc = enc.cuda().eval()
    enc.use_cuda_graph = True
    plan = bench.label_plan(L, B, model["vocab"], seed=7)
    enc.ctc_logit_bump = (plan.to(torch.int32).cuda().contiguous(), bench.CTC_MARGIN)
    x, lens = bench.make_batch(lengths, model["feat_dim"], 1234)
    xn = ops.cmvn(x.cuda(), lens.to(torch.int32).cuda())
    outs = {}
    for prec in ("bf16", "fp32"):
        enc.precision = prec
        for _ in range(warmup):
            outs[prec] = enc(xn, lens)
    times = {"bf16": [], "fp32": []}
    for _ in range(3):  # alternate: drift of clocks / neighbours hits both
        for prec in ("bf16", "fp32"):
            enc.precision = prec
            times[prec].append(time_events(lambda: enc(xn, lens), steps))
    # parity of each precision against the fp32 CPU oracle on the first utterances
    sd = {k: v.detach().float().cpu() for k, v in enc.state_dict().items()}
    xr = torch.zeros(n_ref, T, model["feat_dim"])
    for b in range(n_ref):
        xr[b, : lengths[b]] = O.cmvn(x[b, : lengths[b]])
    ref = O.encoder_forward(sd, model, xr, lens[:n_ref], ctc_logits_hook=O.bump_hook(plan[:, :n_ref],
                                                                                      bench.CTC_MARGIN))
    nl = ref["src_lengths"].tolist()
    res = dict(config=name, batch="%d utterances, %d frames" % (B, sum(lengths)))
    for prec in ("bf16", "fp32"):
        o = outs[prec]
        same_len = o.src_lengths.cpu()[:n_ref].tolist() == nl
        rep = parity_report(o.encoder_out[:, :n_ref].float().cpu(), ref["encoder_out"], nl) if same_len else {}
        sec = sorted(times[prec])[1]
        res[prec] = dict(frames_per_s=round(sum(lengths) / sec, 1), ms_per_step=round(sec * 1e3, 3),
                         lengths_exact=same_len, parity_vs_fp32_oracle=dict(utterances=n_ref, **rep))
    res["fp32_over_bf16_time"] = round(res["bf16"]["frames_per_s"] / res["fp32"]["frames_per_s"], 2)
    ns = argparse.Namespace(config=name)
    res["reference_fp32_eager_same_gpu"] = bench.reference_gpu_eager(ns, enc.state_dict(), plan)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg1,cfg2")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--ref-utts", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_precision: needs a B200 (no CPU timing)")
    res = dict(card=card(), timing="CUDA events, median of 3 alternating windows of --steps forwards",
               gemm=gemm_rate(args.steps),
               configs=[run_config(c, args.steps, args.warmup, args.ref_utts) for c in args.configs.split(",")])
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
