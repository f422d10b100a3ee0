"""The encoder backward at the cfg4 encoder shape with different gradient requests, and the conv1 data-gradient
kernel against its HBM floor.

    python scripts/bench_input_grad.py [--steps 20] [--warmup 3]

Shape: the cfg4 encoder (11L d512 h8 ffn2048, log penalty, CTC compression avg at layer 8, batch 64 x 1500 x 40),
in eval() (running statistics, no dropout) so that the arms differ only in what the backward computes, with
bench.py's run-structured CTC logit injection.  One step:
encoder forward (untimed) -> backward of <encoder_out, R> + <ctc_out, Rc>; CUDA events around the backward.  Arms:
  (a) every parameter trainable, no input gradient (the full training backward);
  (b) every parameter frozen, input gradient only (attribution);
  (c) only the top 3 layers, the final LayerNorm and ctc_fc trainable (fine-tuning a pretrained encoder's top).
After warm-up the arms alternate step by step.  (d) times ``ops.conv1_dgrad`` alone on the cfg4 gradient shape,
rotating over four dz1 buffers (4 x 123 MB, larger than the 126 MB L2) so each call reads from HBM, and compares
it with the bytes it must move at the data-sheet 7.7 TB/s.  Prints the card's name, power limit and max SM clock."""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "fbk-fairseq-st_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import bench  # noqa: E402
from fbkst_b200 import ops  # noqa: E402
from fbkst_b200.config import build_encoder  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # NVIDIA HGX B200 data sheet, one GPU


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "nvidia-smi failed: " + r.stdout.strip()


def summary(t):
    return "median %8.3f ms  mean %8.3f  min %8.3f  max %8.3f" % (statistics.median(t), statistics.mean(t), min(t),
                                                                   max(t))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="timed backwards per arm (alternated)")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps per arm first")
    ap.add_argument("--kernel-iters", type=int, default=200, help="timed conv1_dgrad calls")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_input_grad: needs a CUDA device")
    cfg = bench.CONFIGS["cfg4"]["model"]
    lengths = bench.CONFIGS["cfg4"]["lengths"]
    enc = build_encoder(cfg)  # eval()
    x, lens = bench.make_batch(lengths, cfg["feat_dim"], seed=1)
    x, lens = x.cuda(), lens.cuda()
    # bench.py's run-structured CTC logit injection: the compressed layers see the lengths a trained model gives
    L = ((max(lengths) + 1) // 2 + 1) // 2
    plan = bench.label_plan(L, len(lengths), cfg["vocab"], seed=7).cuda()
    enc.ctc_logit_bump = (plan.to(torch.int32).contiguous(), bench.CTC_MARGIN)
    n_layers = len(enc.layers)
    top = tuple("layers.%d." % i for i in range(n_layers - 3, n_layers)) + ("layer_norm.", "ctc_fc.")
    arms = {
        "a": ("(a) every parameter, no input gradient", lambda n: True, False),
        "b": ("(b) input gradient only, frozen model", lambda n: False, True),
        "c": ("(c) top 3 layers + final LN + ctc_fc", lambda n: n.startswith(top), False),
    }
    g = torch.Generator().manual_seed(2)
    R = Rc = None

    def step(arm):
        nonlocal R, Rc
        _, trainable, want_x = arms[arm]
        for n, p in enc.named_parameters():
            p.requires_grad_(trainable(n))
            p.grad = None
        xd = x.clone().requires_grad_(want_x)
        out = enc(xd, lens)
        if R is None:
            R = (torch.randn(out.encoder_out.shape, generator=g) * 1e-3).cuda()
            Rc = (torch.randn(out.ctc_out.shape, generator=g) * 1e-3).cuda()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        torch.autograd.backward([out.encoder_out, out.ctc_out], [R, Rc])
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e)

    for _ in range(args.warmup):
        for arm in arms:
            step(arm)
    times = {a: [] for a in arms}
    order = list(arms)
    for i in range(args.steps):
        for arm in (order if i % 2 == 0 else order[::-1]):
            times[arm].append(step(arm))
    for p in enc.parameters():
        p.grad = None
    del enc

    # (d) the kernel alone, cold in L2
    C = cfg["conv_channels"]
    B, T, Fd = len(lengths), max(lengths), cfg["feat_dim"]
    T1, F1 = (T + 1) // 2, (Fd + 1) // 2
    dzs = [torch.randn(B, T1, F1, C, device="cuda").bfloat16() for _ in range(4)]
    w1 = torch.randn(C, 9, device="cuda") * 0.3
    for dz in dzs:
        ops.conv1_dgrad(dz, w1, T, Fd)
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(args.kernel_iters):
        ops.conv1_dgrad(dzs[i % 4], w1, T, Fd)
    e.record()
    torch.cuda.synchronize()
    t_kernel = s.elapsed_time(e) / args.kernel_iters * 1e-3
    moved = dzs[0].numel() * 2 + B * T * Fd * 4 + w1.numel() * 4
    floor = moved / HBM_BYTES_PER_S

    print("card: %s" % card())
    print("shape: cfg4 encoder (%dL d%d, ctc-compress %s at layer %d), eval(), batch %d x %d x %d; backward only, "
          "%d alternated steps per arm after %d warm-up steps" %
          (n_layers, cfg["embed_dim"], cfg["ctc_strategy"], cfg["ctc_layer"], B, T, Fd, args.steps, args.warmup))
    for arm, (name, _, _) in arms.items():
        print("%-42s %s" % (name, summary(times[arm])))
    ta = statistics.median(times["a"])
    for arm in ("b", "c"):
        print("ratio %s/(a) of medians: %.3f" % (arm, statistics.median(times[arm]) / ta))
    print("(d) conv1_dgrad [%d,%d,%d,%d] bf16 -> [%d,%d,%d] fp32: %.2f us/call over %d calls (4 rotating inputs); "
          "%.1f MB moved, %.0f GB/s; data-sheet HBM floor %.2f us (%.0f%% of it)" %
          (B, T1, F1, C, B, T, Fd, t_kernel * 1e6, args.kernel_iters, moved / 1e6, moved / t_kernel / 1e9,
           floor * 1e6, 100.0 * floor / t_kernel))


if __name__ == "__main__":
    main()
