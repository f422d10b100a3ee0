"""The kernels as PyTorch custom operators: ``torch.ops.fbkst.<op>``.

BASELINE.json's north_star asks for the sm_100a kernels "behind a thin C-ABI exposed as PyTorch
custom ops".  The C ABI is ``include/fbkst_b200.h`` (ctypes binding in ``_lib.py``, tensor-level
wrappers in ``ops.py``); this module registers those wrappers with the dispatcher under the
``fbkst`` namespace for the CUDA backend ONLY.  There is deliberately no CPU / Meta / autograd
kernel: calling an op on CPU tensors fails in the dispatcher ("Could not run 'fbkst::...' with
arguments from the 'CPU' backend") instead of silently computing something else.

The encoder itself calls ``ops.*`` directly (one Python frame less per launch; irrelevant once the
forward is replayed from a CUDA graph) -- both routes end in the same ``extern "C"`` entry points.
"""
import torch

from . import ops

_lib = torch.library.Library("fbkst", "DEF")
_EMPTY = {}


def _def(schema, fn):
    _lib.define(schema)
    _lib.impl(schema.split("(")[0], fn, "CUDA")


def _linear(a, w, bias, relu, residual, out_f32):
    return ops.linear(a, w, bias, relu=relu, residual=residual,
                      out_dtype=torch.float32 if out_f32 else torch.bfloat16)


def _layernorm(x, gamma, beta, out_f32, eps):
    return ops.layernorm(x, gamma, beta, out_dtype=torch.float32 if out_f32 else torch.bfloat16, eps=eps)


def _ctc_argmax(logits, lengths, L, B, V, want_prob):
    labels, prob = ops.ctc_argmax(logits, lengths, L, B, V, want_prob)
    if prob is None:
        prob = torch.empty(0, dtype=torch.float32, device=logits.device)
    return labels, prob


def _ctc_segment(labels, top_prob, lengths, strategy, L, B):
    if top_prob is not None and top_prob.numel() == 0:
        top_prob = None
    return ops.ctc_segment(labels, top_prob, lengths, strategy, L, B)


_def("cmvn(Tensor x, Tensor lengths) -> Tensor", lambda x, lengths: ops.cmvn(x, lengths))
_def("conv1_relu_bn(Tensor x, Tensor w, Tensor bias, Tensor scale, Tensor shift) -> Tensor",
     ops.conv1_relu_bn)
_def("conv2_relu_bn(Tensor x, Tensor w_taps, Tensor bias, Tensor scale, Tensor shift) -> Tensor",
     ops.conv2_relu_bn)
_def("linear(Tensor a, Tensor w, Tensor? bias, bool relu, Tensor? residual, bool out_f32) -> Tensor",
     _linear)
_def("layernorm(Tensor x, Tensor gamma, Tensor beta, bool out_f32, float eps) -> Tensor", _layernorm)
_def("attention(Tensor qkv, Tensor lengths, int L, int B, int H, bool log_penalty) -> Tensor",
     lambda qkv, lengths, L, B, H, log_penalty: ops.attention(qkv, lengths, L, B, H, log_penalty))
_def("linear_f32(Tensor a, Tensor w, Tensor? bias, bool relu, Tensor? residual) -> Tensor",
     lambda a, w, bias, relu, residual: ops.linear_f32(a, w, bias, relu=relu, residual=residual))
_def("attention_f32(Tensor qkv, Tensor lengths, int L, int B, int H, bool log_penalty) -> Tensor",
     lambda qkv, lengths, L, B, H, log_penalty: ops.attention_f32(qkv, lengths, L, B, H, log_penalty))
_def("ctc_argmax(Tensor logits, Tensor lengths, int L, int B, int V, bool want_prob) -> (Tensor, Tensor)",
     _ctc_argmax)
_def("ctc_segment(Tensor labels, Tensor? top_prob, Tensor lengths, str strategy, int L, int B)"
     " -> (Tensor, Tensor, Tensor, Tensor, Tensor)", _ctc_segment)
_def("ctc_compress(Tensor x, Tensor seg_id, Tensor seg_start, Tensor weight, Tensor lengths,"
     " Tensor new_len, Tensor max_new, int L, int B) -> Tensor",
     lambda x, seg_id, seg_start, weight, lengths, new_len, max_new, L, B:
     ops.ctc_compress(x, seg_id, seg_start, weight, lengths, new_len, max_new, L, B))
_def("lengths_to_mask(Tensor lengths, int L) -> Tensor", lambda lengths, L: ops.lengths_to_mask(lengths, L)[0])


def _xattn(q, kv, mask, row_map, tgt_len, H, weights):
    S, U = kv.shape[0], kv.shape[1]
    out, w = ops.xattn(q, kv, mask, row_map, S, U, row_map.numel(), tgt_len, H, weights=weights)
    if w is None:
        w = torch.empty(0, dtype=torch.float32, device=q.device)
    return out, w


_def("xattn(Tensor q, Tensor kv, Tensor? mask, Tensor row_map, int tgt_len, int H, int weights)"
     " -> (Tensor, Tensor)", _xattn)

OPS = ["cmvn", "conv1_relu_bn", "conv2_relu_bn", "linear", "layernorm", "attention", "linear_f32",
       "attention_f32", "ctc_argmax",
       "ctc_segment", "ctc_compress", "lengths_to_mask", "xattn"]
