"""Host side of ``criterion.CtcProjection``: locating the CTC criterion's ``fc_out`` on a stand-in module tree (the
reference criterion's ``ctc_aware_model.fc_out``) and swapping it without changing parameters or state-dict keys."""
import pytest
import torch

from fbkst_b200 import criterion as C


class _Wrapper(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.fc_out = torch.nn.Linear(16, 11)
        self.other = torch.nn.Linear(16, 4)


class _Criterion(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.ctc_aware_model = _Wrapper()
        self.real_criterion = torch.nn.Module()


def test_locates_and_swaps_the_single_fc_out():
    crit = _Criterion()
    lin = crit.ctc_aware_model.fc_out
    keys = {k: v for k, v in crit.state_dict().items()}
    params = dict(crit.named_parameters())
    parent, attr, mod = C.find_ctc_projection(crit)
    assert parent is crit.ctc_aware_model and attr == "fc_out" and mod is lin
    proj = C.install_ctc_projection(crit)
    assert isinstance(crit.ctc_aware_model.fc_out, C.CtcProjection) and crit.ctc_aware_model.fc_out is proj
    assert proj.weight is lin.weight and proj.bias is lin.bias
    assert (proj.in_features, proj.out_features) == (16, 11)
    assert list(crit.state_dict().keys()) == list(keys.keys())
    assert all(torch.equal(crit.state_dict()[k], v) for k, v in keys.items())
    assert {n: id(p) for n, p in crit.named_parameters()} == {n: id(p) for n, p in params.items()}
    crit.load_state_dict(keys, strict=True)
    assert C.install_ctc_projection(crit) is proj  # idempotent
    crit.half()  # fairseq --fp16: the same Parameter objects are converted in place
    assert proj.weight is lin.weight and proj.weight.dtype == torch.float16


def test_fc_out_at_the_top_level():
    m = torch.nn.Module()
    m.fc_out = torch.nn.Linear(8, 5)
    parent, attr, _ = C.find_ctc_projection(m)
    assert parent is m and attr == "fc_out"


def test_no_fc_out_raises():
    m = torch.nn.Module()
    m.proj = torch.nn.Linear(8, 5)
    m.fc_out = torch.nn.Conv1d(8, 5, 1)  # not a Linear
    with pytest.raises(ValueError, match="exactly one.*found 0"):
        C.find_ctc_projection(m)
    with pytest.raises(ValueError, match="found 0"):
        C.install_ctc_projection(m)


def test_two_fc_out_raise():
    crit = _Criterion()
    crit.real_criterion.fc_out = torch.nn.Linear(16, 3)
    with pytest.raises(ValueError, match=r"found 2.*ctc_aware_model\.fc_out.*real_criterion\.fc_out"):
        C.install_ctc_projection(crit)
    assert isinstance(crit.ctc_aware_model.fc_out, torch.nn.Linear)  # nothing swapped


def test_wraps_only_a_linear_and_has_no_cpu_path():
    with pytest.raises(TypeError):
        C.CtcProjection(torch.nn.Conv1d(8, 5, 1))
    proj = C.CtcProjection(torch.nn.Linear(8, 5))
    with pytest.raises(ValueError, match="CUDA"):
        proj(torch.randn(3, 2, 8))
