"""CPU checks of the ``precision`` switch of the encoder (no GPU needed)."""
import pytest

import bench
from fbkst_b200.config import build_encoder


def _enc(**kw):
    return build_encoder(dict(bench.CONFIGS["cfg1"]["model"], **kw), None, device="cpu")


def test_default_is_bf16():
    enc = _enc()
    assert enc.precision == "bf16"
    assert enc.ctc_fc.precision == "bf16"


def test_config_and_setter_select_fp32():
    enc = _enc(precision="fp32")
    assert enc.precision == "fp32" and enc.ctc_fc.precision == "fp32"
    enc.precision = "bf16"
    assert enc.ctc_fc.precision == "bf16"


@pytest.mark.parametrize("bad", ["fp16", "FP32", "tf32", None, 32])
def test_unknown_precision_raises(bad):
    enc = _enc()
    with pytest.raises(ValueError, match="precision"):
        enc.precision = bad
    assert enc.precision == "bf16"
    with pytest.raises(ValueError, match="precision"):
        _enc(precision=bad)


def test_precision_is_part_of_the_graph_key():
    enc = _enc()
    k_bf16 = enc._graph_key(2, 100, 40, "cuda:0")
    enc.precision = "fp32"
    k_f32 = enc._graph_key(2, 100, 40, "cuda:0")
    assert k_bf16 != k_f32 and "fp32" in k_f32 and "bf16" in k_bf16


def test_training_in_fp32_raises_before_any_kernel():
    import torch
    enc = _enc(precision="fp32").train()
    with pytest.raises((NotImplementedError, RuntimeError)):
        enc(torch.zeros(1, 40, 40), torch.tensor([40]))
