"""GPU parity of the device SpecAugment / TimeStretch (SURVEY 8f N3), through the C ABI.

  * golden vectors produced by the LIVE reference modules under fixed seeds (bit-exact: the ops only
    move or zero fp32 values, and the stretch indices are an integer contract);
  * the CPU oracle on seeded inputs, including odd feature widths and full-size batches."""
import os
import random

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import augment_oracle as A  # noqa: E402  (checker only)
from oracle.golden import load as load_golden  # noqa: E402


def seed(s):
    random.seed(s)
    np.random.seed(s)


def dev():
    return torch.device("cuda:0")


def test_specaugment_golden(golden_dir):
    from fbkst_b200.augment import SpecAugment
    golden = load_golden(os.path.join(golden_dir, "augment.pt"))["spec"]
    for name, c in golden.items():
        seed(c["seed"])
        x = c["x"].to(dev())
        out = SpecAugment(*c["pars"])({"net_input": {"src_tokens": x}})["net_input"]["src_tokens"]
        assert torch.equal(out.cpu(), c["ref"]), name
        assert out.data_ptr() == x.data_ptr()  # in place


def test_time_stretch_golden(golden_dir):
    from fbkst_b200.augment import TimeStretch
    golden = load_golden(os.path.join(golden_dir, "augment.pt"))["stretch"]
    for name, c in golden.items():
        seed(c["seed"])
        m = TimeStretch(*c["pars"])
        batch = {"id": torch.arange(len(c["lengths"])), "target": "kept",
                 "net_input": {"src_tokens": c["x"].to(dev()), "src_lengths": torch.tensor(c["lengths"]).to(dev()),
                               "prev_output_tokens": "kept"}}
        nb = m(batch)
        assert nb["net_input"]["src_lengths"].tolist() == c["ref_lengths"], name
        assert nb["net_input"]["src_lengths"].dtype == torch.long and nb["net_input"]["src_lengths"].is_cuda
        assert torch.equal(m.last_ids.cpu().long(), c["ref_ids"]), name
        assert torch.equal(nb["net_input"]["src_tokens"].cpu(), c["ref"]), name
        assert nb["target"] == "kept" and nb["net_input"]["prev_output_tokens"] == "kept"
        assert batch["net_input"]["src_tokens"].shape == c["x"].shape  # the input batch is not modified


@pytest.mark.parametrize("F,B,T", [(40, 64, 1500), (80, 8, 6000), (83, 3, 257), (1, 2, 33)])
def test_augment_vs_oracle(F, B, T):
    from fbkst_b200.augment import SpecAugment, TimeStretch
    g = torch.Generator().manual_seed(F * 7 + B)
    lengths = sorted([int(v) for v in torch.randint(max(T // 4, 1), T + 1, (B,), generator=g)], reverse=True)
    lengths[0] = T
    x = torch.randn(B, T, F, generator=g) + 2.5
    for b, n in enumerate(lengths):
        x[b, n:] = 0
    for s, pars in ((31, (13, 13, 2, 2, 1.0)), (32, (27, 100, 1, 2, 0.7))):
        pars = (min(pars[0], F),) + pars[1:]
        seed(s)
        want = A.specaugment_batch(x.numpy(), *pars)
        seed(s)
        got = SpecAugment(*pars)({"net_input": {"src_tokens": x.to(dev())}})["net_input"]["src_tokens"]
        assert np.array_equal(got.cpu().numpy(), want)
    for s, pars in ((41, (1.0, 1, 0.8, 1.25)), (42, (0.8, 7, 0.8, 1.25)), (43, (1.0, 50, 0.5, 1.5))):
        seed(s)
        want, nl, ids = A.time_stretch_batch(x.numpy(), lengths, *pars)
        seed(s)
        m = TimeStretch(*pars)
        nb = m({"net_input": {"src_tokens": x.to(dev()), "src_lengths": torch.tensor(lengths)}})
        assert nb["net_input"]["src_lengths"].tolist() == nl
        for b, i in enumerate(ids):
            assert np.array_equal(m.last_ids[b, :len(i)].cpu().numpy(), i), b
            assert (m.last_ids[b, len(i):] == -1).all()
        assert np.array_equal(nb["net_input"]["src_tokens"].cpu().numpy(), want)


def test_time_stretch_everything_dropped():
    """w = 1 with high < 1 keeps no frame at all (int(s) = 0 for every window): empty batch like the
    reference's fancy index with an empty list."""
    from fbkst_b200.augment import TimeStretch
    seed(0)
    x = torch.ones(2, 20, 4, device=dev())
    nb = TimeStretch(1.0, 1, 0.5, 0.9)({"net_input": {"src_tokens": x, "src_lengths": torch.tensor([20, 12])}})
    assert nb["net_input"]["src_lengths"].tolist() == [0, 0]
    assert tuple(nb["net_input"]["src_tokens"].shape) == (2, 0, 4)
