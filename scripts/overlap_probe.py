#!/usr/bin/env python
"""Does running two encoder forwards on two CUDA streams fill the per-kernel tail waves?

Every kernel of the step is a persistent grid of <=148 CTAs (or 296 for attention), so the last wave of
each launch leaves SMs idle (tile counts at cfg2: qkv 7.6 waves, fc1 10.2, out_proj/fc2 2.5, attention
5.2).  With two independent batches in flight on two streams the CTAs of one stream's kernel start on
the SMs the other stream's kernel has already left.  Diagnostic only: prints ms/step (device, CUDA
events across both streams) for 1 stream and 2 streams.
"""
import copy
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import torch  # noqa: E402
from fbkst_b200 import ops  # noqa: E402
from fbkst_b200.config import build_encoder  # noqa: E402


def smi():
    o = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=clocks.sm,power.draw",
                        "--format=csv,noheader,nounits"], capture_output=True, text=True).stdout
    return o.strip()


def main():
    n_streams = int(sys.argv[1]) if len(sys.argv) > 1 else 2
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 200
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    cfg = bench.CONFIGS[os.environ.get("CFG", "cfg2")]
    model, lengths = cfg["model"], cfg["lengths"]
    B, T, Fd = len(lengths), max(lengths), model["feat_dim"]
    torch.manual_seed(0)
    enc0 = build_encoder(model, None, device="cpu")
    bench.randomise_norm_stats(enc0, 1)
    L = ((T + 1) // 2 + 1) // 2
    plan = bench.label_plan(L, B, model["vocab"], seed=7).to(dev)

    def bump(mod, inp, out):
        out.scatter_add_(2, plan.unsqueeze(-1),
                         torch.full((L, B, 1), bench.CTC_MARGIN, dtype=out.dtype, device=out.device))
    encs = []
    for s in range(n_streams):
        e = copy.deepcopy(enc0).to(dev).eval()
        e.use_cuda_graph = True
        e.ctc_fc.register_forward_hook(bump)
        encs.append(e)
    devb = [(x.to(dev), l) for x, l in (bench.make_batch(lengths, Fd, 1234 + i) for i in range(4))]
    len32 = torch.tensor(lengths, dtype=torch.int32, device=dev)
    streams = [torch.cuda.Stream(dev) for _ in range(n_streams)]

    def body(i):
        """the graph body only (no end-of-forward host sync): CMVN + replay"""
        e = encs[i % n_streams]
        x, l = devb[i % 4]
        xn = ops.cmvn(x, len32)
        return e._replay(xn, [L] * B, B, T, Fd, L)

    for i in range(2 * n_streams):  # capture + warm-up
        with torch.cuda.stream(streams[i % n_streams]):
            encs[i % n_streams](ops.cmvn(devb[i % 4][0], len32), devb[i % 4][1])
    torch.cuda.synchronize()
    res = dict(n_streams=n_streams, steps=steps)
    for rep in range(2):
        s0, e0 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        main_s = torch.cuda.current_stream()
        torch.cuda._sleep(int(5e-3 * 1.9e9))
        s0.record(main_s)
        for st in streams:
            st.wait_event(s0)
        for i in range(steps):
            with torch.cuda.stream(streams[i % n_streams]):
                body(i)
        for st in streams:
            main_s.wait_stream(st)
        e0.record(main_s)
        torch.cuda.synchronize()
        res["ms_per_step_rep%d" % rep] = s0.elapsed_time(e0) / steps
        res["smi_rep%d" % rep] = smi()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
