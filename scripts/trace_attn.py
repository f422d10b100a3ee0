"""Timeline of CTA 0 of the wide attention kernel (debug hook fbkst_debug_set_attention_wide_trace)."""
import ctypes
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "fbk-fairseq-st_b200"))
from fbkst_b200 import _lib, ops  # noqa: E402

lib = _lib.load()
lib.fbkst_debug_set_attention_wide_trace.argtypes = [ctypes.c_void_p]
d = torch.device("cuda:0")
L, B, H = 375, 64, 8
qkv = (torch.randn(L * B, 3 * H * 64, device=d) * 0.7).bfloat16()
lengths = torch.full((B,), L, dtype=torch.int32, device=d)
q_limit = None
if os.environ.get("FBKST_TRACE_POST"):  # the in-step shape after CTC compression: worst-case grid, short utterances
    lens = [120 + (i * 7) % 13 for i in range(B)]
    lengths = torch.tensor(lens, dtype=torch.int32, device=d)
    q_limit = torch.tensor([max(lens)], dtype=torch.int32, device=d)
_attention = ops.attention
ops.attention = lambda *a, **k: _attention(*a, q_limit=q_limit, **k)
for _ in range(3):
    ops.attention(qkv, lengths, L, B, H, True)
buf = torch.zeros(64 * 16, dtype=torch.int64, device=d)
assert lib.fbkst_debug_set_attention_wide_trace(buf.data_ptr()) == 0
ops.attention(qkv, lengths, L, B, H, True)
torch.cuda.synchronize()
lib.fbkst_debug_set_attention_wide_trace(None)
t = buf.view(64, 16).cpu()
t0 = int(t[t > 0].min())
order = [(14, "tma:K"), (11, "mma:QK"), (0, "s_full"), (1, "S_regs"), (2, "guard"), (3, "P_done"), (4, "P_free"),
         (5, "p_full"), (12, "mma:PV"), (9, "last_pv"), (10, "stored")]
print("tile " + " ".join("%9s" % n for _, n in order))
for i in range(40):
    print("%4d " % i + " ".join("%9d" % (int(t[i][k]) - t0 if t[i][k] > 0 else -1) for k, _ in order))
