"""ctypes binding of ``libfbkst_b200.so`` (declared in ``include/fbkst_b200.h``)."""
import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfbkst_b200.so")

ERR_ARG, ERR_CUDA, ERR_OOM = -1, -2, -3
BF16, F32 = 0, 1
CTC_STRATEGY = {"avg": 0, "weighted": 1, "softmax": 2}
EPI_RELU, EPI_OUT_F32, EPI_ROW_REMAP, EPI_POSEMB, EPI_AB_F16 = 1, 2, 4, 8, 16
SA_INCREMENTAL, SA_FULL, SA_CAUSAL = 0, 1, 2

P, I, I64, F, U64 = c_void_p, c_int, c_int64, c_float, c_uint64

# name -> argtypes; every entry point returns int (0 = ok) unless listed in _RESTYPES
SIGNATURES = {
    "fbkst_abi_version": [],
    "fbkst_device_ok": [],
    "fbkst_cmvn_f32": [P, P, P, I, I, I, P, P],
    "fbkst_collate_cmvn_f32": [P, P, P, P, I, I, I, I, P, P],
    "fbkst_conv1_relu_bn": [P, P, P, P, P, P, I, I, I, I, P],
    "fbkst_conv2_relu_bn": [P, P, P, P, P, P, I, I, I, I, P],
    "fbkst_conv1_relu_bn_planes": [P, P, P, P, P, P, I, I, I, I, P],
    "fbkst_conv2_relu_bn_planes": [P, P, P, P, P, P, I, I, I, I, P],
    "fbkst_linear_bf16": [P, I64, P, I64, P, P, I64, P, I64, I, I, I, I, I, I, P, P, I, P],
    "fbkst_linear_ln_bf16": [P, I64, P, I64, P, P, I64, P, I64, I, I, I, I, P, F, P, I64, P, P, I, P],
    "fbkst_row_stats_cast": [P, P, P, I, I, P, I, P],
    "fbkst_embed_remap_stats": [P, P, I64, P, P, P, P, I, I, I, P],
    "fbkst_layernorm": [P, P, P, P, I, I, I, F, P, I, P],
    "fbkst_attention_fwd": [P, P, P, I, I, I, I, P],
    "fbkst_attention_fwd_limited": [P, P, P, I, I, I, I, P, P],
    "fbkst_sinusoidal_table": [P, I, I, P],
    "fbkst_lengths_to_mask": [P, P, P, I, I, P],
    "fbkst_subsample_lengths": [P, I, P, I, I, P],
    "fbkst_linear_argmax_f32": [P, I64, P, I64, P, P, I64, I, I, I, P, F, I, P, P, I, P],
    "fbkst_ctc_argmax_merge": [P, I, P, I64, I, P, P, P, P, I, I, P],
    "fbkst_ctc_argmax": [P, I, I64, P, P, P, I, I, I, P],
    "fbkst_ctc_argmax_lse": [P, I, I64, P, P, P, P, I, I, I, P],
    "fbkst_ctc_uer": [P, P, P, I64, P, I, P, P, P, I, I, I, P],
    "fbkst_ctc_loss_fwd": [P, I, I64, P, P, P, I64, P, I, P, P, I, I, I, I, P],
    "fbkst_ctc_segment": [P, P, P, I, P, P, P, P, P, I, I, P],
    "fbkst_ctc_compress": [P, P, P, P, P, P, P, P, I, I, I, P],
    "fbkst_specaugment_f32": [P, P, I, I, I, I, I, P],
    "fbkst_time_stretch_f32": [P, P, I, P, P, I, I, I, I, P],
    "fbkst_xattn_fwd": [P, P, P, P, P, P, P, I, I, I, I, I, I, P],
    "fbkst_xattn_fwd_f32": [P, P, P, P, P, P, P, I, I, I, I, I, I, P],
    "fbkst_dec_self_attn_fwd": [P, I64, P, P, P, P, P, I, I, I, I, I, I, I, P],
    "fbkst_dec_self_attn_fwd_f32": [P, I64, P, P, P, P, P, I, I, I, I, I, I, I, P],
    "fbkst_cast_bf16": [P, P, I64, F, P],
    "fbkst_prep_conv2_weight": [P, P, I, P],
    "fbkst_prep_fc3_weight": [P, P, I, I, I, P],
    "fbkst_prep_bn_affine": [P, P, P, P, F, P, P, I, P],
    # fp32-accurate inference path (split TF32)
    "fbkst_linear_tf32x3": [P, I64, P, I64, P, P, P, P, I64, P, I64, I, I, I, I, P, I, P],
    "fbkst_attention_tf32x3": [P, P, P, I, I, I, I, P, P],
    "fbkst_conv1_relu_bn_f32": [P, P, P, P, P, P, I, I, I, I, P],
    "fbkst_conv2_im2col_f32": [P, P, I, I, I, I, P],
    # training side
    "fbkst_dropout_add_ln": [P, P, P, P, P, P, F, I, I, F, U64, I, P],
    "fbkst_ln_bwd_blocks": [I],
    "fbkst_ln_bwd": [P, P, P, P, I, P, F, I, I, P],
    "fbkst_grad_prep": [P, I, I64, P, I64, F, I, I, P, I64, I, P, I64, P, I, I, I, F, U64, I, I, P],
    "fbkst_reduce_sum": [P, I, I64, I, I, I64, P, I64, F, P],
    "fbkst_linear_wgrad_bf16": [P, I64, P, I64, P, P, I64, I, I, I, P],
    "fbkst_linear_wgrad_nt": [P, I64, P, I64, I, P, P, I64, I, I, I, P],
    "fbkst_linear_wgrad_slices_bf16": [P, I64, P, I64, P, I, I, I, P, P],
    "fbkst_reduce_sum_batch": [P, I, P],
    "fbkst_prep_batch": [P, I, P],
    "fbkst_attention_train_fwd": [P, P, P, P, I, I, I, I, F, U64, I, P],
    "fbkst_attn_delta": [P, P, P, I, I, P],
    "fbkst_attention_train_bwd": [P, P, P, P, P, P, I, I, I, I, F, U64, I, P],
    "fbkst_ctc_compress_bwd": [P, P, P, P, I, I, I, P],
    "fbkst_dropout_inplace": [P, I, I64, F, U64, I, P],
    "fbkst_ctc_loss_bwd": [P, I, I64, P, P, P, I64, P, I, P, P, P, I64, I, I, I, I, P],
    "fbkst_bn_partial_blocks": [],
    "fbkst_bn_batch_stats": [P, I64, I, P, P, F, F, P, P, P, P, P, P, P, P],
    "fbkst_bn_apply": [P, P, P, P, I64, I, F, U64, I, P],
    "fbkst_bn_relu_bwd": [P, P, P, P, P, I, P, P, P, I64, I, F, U64, I, P],
    "fbkst_conv2_im2col_t": [P, P, I64, I, I, I, I, P],
    "fbkst_conv2_col2im": [P, P, I, I, I, I, P],
    "fbkst_conv1_wgrad": [P, P, P, P, I, I, I, I, P],
}
_RESTYPES = {"fbkst_linear_wgrad_workspace": (c_int64, [I, I, I]),
             "fbkst_ctc_loss_bwd_workspace": (c_int64, [I, I, I])}

_lib = None


def load():
    """Load the shared library (no GPU needed); raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "fbkst_b200: %s is missing -- build it with `python fbk-fairseq-st_b200/build.py` "
            "(there is no CPU / PyTorch fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    lib.fbkst_last_error.restype = c_char_p
    lib.fbkst_last_error.argtypes = []
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = c_int
    for name, (restype, argtypes) in _RESTYPES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype
    _lib = lib
    return lib


def check(rc):
    if rc == 0:
        return
    msg = load().fbkst_last_error().decode("utf-8", "replace")
    if rc == ERR_OOM:
        raise RuntimeError("CUDA out of memory in fbkst_b200: " + msg)
    if rc == ERR_ARG:
        raise ValueError("fbkst_b200: " + msg)
    raise RuntimeError("fbkst_b200: " + msg)


_device_checked = False


def require_device():
    """The product path needs the library AND a compute-capability-10.x device."""
    global _device_checked
    lib = load()
    if not _device_checked:
        if not lib.fbkst_device_ok():
            raise RuntimeError("fbkst_b200: no sm_100 (B200) CUDA device visible; this package has "
                               "no CPU fallback")
        _device_checked = True
    return lib
