"""CTC-multitask training step WITHOUT compression at the cfg4 encoder shape: the two ways of projecting the CTC
state, timed against each other.

    python scripts/bench_ctc_multitask.py [--steps 20] [--warmup 3]

Shape: the cfg4 encoder (11L d512 h8 ffn2048, log penalty, batch 64 x 1500 x 40, V = 8005) with no CTC compression,
in train() (dropout, BatchNorm batch statistics).  One step: encoder forward (return_all_hiddens) -> CTC loss on
encoder_states[7] (CTC at layer 8) -> a stand-in decoder loss <encoder_out, R> -> backward.  Arms:
  (a) criterion.CtcProjection + ctc_loss_train: tcgen05 projection, its backward inside the CTC loss node;
  (b) nn.Linear under bf16 autocast (cuBLAS) feeding criterion.CtcLossFn (the projection's backward on autograd).
Both use the same parameters and the same dropout seeds.  After warm-up the arms alternate step by step; CUDA events
around every step.  Prints ms/step per arm with the card's name, power limit and max SM clock."""
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
from fbkst_b200 import criterion as C  # noqa: E402
from fbkst_b200.config import build_encoder  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "nvidia-smi failed: " + r.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="timed steps per arm (alternated)")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps per arm first")
    ap.add_argument("--ctc-layer", type=int, default=8)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ctc_multitask: needs a CUDA device")
    cfg = dict(bench.CONFIGS["cfg4"]["model"], ctc_layer=0)  # no compression
    lengths = bench.CONFIGS["cfg4"]["lengths"]
    V, D, k = cfg["vocab"], cfg["embed_dim"], args.ctc_layer
    enc = build_encoder(cfg).train()
    for p in enc.parameters():
        p.requires_grad_(True)
    torch.manual_seed(0)
    lin = torch.nn.Linear(D, V).cuda()
    proj = C.CtcProjection(lin)  # same Parameter objects: both arms train the same weights
    x, lens = bench.make_batch(lengths, cfg["feat_dim"], seed=1)
    x, lens = x.cuda(), lens.cuda()
    B = len(lengths)
    L = ((max(lengths) + 1) // 2 + 1) // 2
    g = torch.Generator().manual_seed(2)
    blank = V - 1
    U = 60
    tg = torch.randint(0, V - 1, (B, U), generator=g).cuda()
    tl = torch.full((B,), U, dtype=torch.int32).cuda()
    il = torch.full((B,), L, dtype=torch.int32).cuda()
    R = (torch.randn(L, B, D, generator=g) * 1e-3).cuda()
    params = list(enc.parameters()) + list(lin.parameters())

    def step(arm, seed):
        torch.manual_seed(seed)  # same dropout masks in both arms
        out = enc(x, lens, return_all_hiddens=True)
        state = out.encoder_states[k - 1]
        if arm == "a":
            loss_ctc = C.ctc_loss_train(proj(state), None, tg, tl, blank)[0]
        else:
            with torch.autocast("cuda", dtype=torch.bfloat16):
                logits = lin(state)
            loss_ctc = C.CtcLossFn.apply(logits, il, tg, tl, blank)[0]
        loss = loss_ctc + (out.encoder_out * R).sum()
        loss.backward()
        for p in params:
            p.grad = None
        return loss_ctc

    arms = ("a", "b")
    for i in range(args.warmup):
        for arm in arms:
            step(arm, 100 + i)
    torch.cuda.synchronize()
    times = {a: [] for a in arms}
    losses = {a: [] for a in arms}
    for i in range(args.steps):
        for arm in (arms if i % 2 == 0 else arms[::-1]):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            lc = step(arm, 1000 + i)
            e.record()
            torch.cuda.synchronize()
            times[arm].append(s.elapsed_time(e))
            losses[arm].append(lc.item())
    print("card: %s" % card())
    print("shape: cfg4 encoder without compression, train(), batch %d x %d x %d, V = %d, CTC loss on "
          "encoder_states[%d]; %d alternated steps per arm after %d warm-up steps" %
          (B, max(lengths), cfg["feat_dim"], V, k - 1, args.steps, args.warmup))
    names = {"a": "(a) CtcProjection, backward in the CTC loss node",
             "b": "(b) nn.Linear under bf16 autocast -> CtcLossFn"}
    for arm in arms:
        t = times[arm]
        print("%-52s median %8.2f ms/step  mean %8.2f  min %8.2f  max %8.2f" %
              (names[arm], statistics.median(t), statistics.mean(t), min(t), max(t)))
    print("ratio (b)/(a) of medians: %.3f" % (statistics.median(times["b"]) / statistics.median(times["a"])))
    d = max(abs(a - b) / abs(b) for a, b in zip(losses["a"], losses["b"]))
    print("CTC loss, same step and seed: max relative difference between the arms %.2e" % d)


if __name__ == "__main__":
    main()
