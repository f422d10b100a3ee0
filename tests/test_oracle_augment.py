"""CPU checks for the next row N3 (SpecAugment / TimeStretch):
  * the oracle restatement against the golden vectors produced by the LIVE reference modules;
  * the oracle against the live reference itself where /root/reference is mounted;
  * the product's HOST logic (RNG draws -> band / window tables) against the same golden vectors --
    the device kernels that consume the tables are checked in tests/test_gpu_augment.py."""
import os
import random

import numpy as np
import pytest
import torch

from oracle import augment_oracle as A
from oracle.golden import load as load_golden
from oracle import ref_loader


@pytest.fixture(scope="module")
def golden(golden_dir):
    return load_golden(os.path.join(golden_dir, "augment.pt"))


def seed(s):
    random.seed(s)
    np.random.seed(s)


def test_spec_oracle_matches_golden(golden):
    for name, c in golden["spec"].items():
        seed(c["seed"])
        y = A.specaugment_batch(c["x"].numpy(), *c["pars"])
        assert np.array_equal(y, c["ref"].numpy()), name


def test_stretch_oracle_matches_golden(golden):
    for name, c in golden["stretch"].items():
        seed(c["seed"])
        rate, w, low, high = c["pars"]
        y, nl, ids = A.time_stretch_batch(c["x"].numpy(), c["lengths"], rate, w, low, high)
        assert nl == c["ref_lengths"], name
        for b, i in enumerate(ids):
            assert np.array_equal(i, c["ref_ids"][b, :len(i)].numpy()), (name, b)
        assert np.array_equal(y, c["ref"].numpy()), name


def test_linspace_round_matches_torch():
    rng = random.Random(0)
    for _ in range(4000):
        w = rng.choice([1, 2, 3, 5, 7, 8, 16, 31, 64, 100, 200])
        start = w * rng.randint(0, 6000 // w)
        end = start + rng.randint(0, w - 1)
        steps = rng.randint(0, int(2.0 * w) + 1)
        want = torch.round(torch.linspace(start, end, steps)).long().numpy()
        assert np.array_equal(A.linspace_round(start, end, steps), want), (start, end, steps)


@pytest.mark.reference
@pytest.mark.skipif(not ref_loader.available(), reason="reference tree not mounted")
def test_oracle_matches_live_reference():
    ref_loader.load()
    from examples.speech_recognition.modules.specaugment import SpecAugment
    from examples.speech_recognition.modules.time_stretch import TimeStretch
    g = torch.Generator().manual_seed(5)
    lengths = [70, 55, 31, 8]
    x = torch.randn(4, 70, 12, generator=g) + 2.0
    for b, n in enumerate(lengths):
        x[b, n:] = 0
    for s, pars in ((1, (5, 20, 2, 1, 1.0)), (2, (12, 100, 1, 3, 0.6))):
        seed(s)
        want = SpecAugment(*pars)({"net_input": {"src_tokens": x.clone()}})["net_input"]["src_tokens"]
        seed(s)
        assert np.array_equal(A.specaugment_batch(x.numpy(), *pars), want.numpy())
    for s, pars in ((3, (1.0, 3, 0.8, 1.25)), (4, (0.5, 1, 0.8, 1.25)), (5, (1.0, 16, 0.6, 1.7))):
        seed(s)
        nb = TimeStretch(*pars)({"net_input": {"src_tokens": x.clone(), "src_lengths": torch.tensor(lengths)}})
        seed(s)
        y, nl, _ = A.time_stretch_batch(x.numpy(), lengths, *pars)
        assert nl == nb["net_input"]["src_lengths"].tolist()
        assert np.array_equal(y, nb["net_input"]["src_tokens"].numpy())


# ---- product host logic (no GPU): the tables the kernels consume ------------------------------------

def apply_bands(x, bands, n_freq):
    y = x.copy()
    for b in range(x.shape[0]):
        for i, (s, w) in enumerate(bands[b]):
            if i < n_freq:
                y[b, :, s:s + w] = 0
            else:
                y[b, s:s + w, :] = 0
    return y


def test_host_bands_reproduce_the_reference_masks(golden):
    from fbkst_b200.augment import SpecAugment
    for name, c in golden["spec"].items():
        seed(c["seed"])
        m = SpecAugment(*c["pars"])
        x = c["x"].numpy()
        bands = m.draw_bands(*x.shape)
        assert bands.dtype == np.int32 and bands.shape == (x.shape[0], c["pars"][2] + c["pars"][3], 2)
        assert np.array_equal(apply_bands(x, bands, c["pars"][2]), c["ref"].numpy()), name


def test_host_windows_reproduce_the_reference_indices(golden):
    from fbkst_b200.augment import TimeStretch
    for name, c in golden["stretch"].items():
        seed(c["seed"])
        m = TimeStretch(*c["pars"])
        windows, owner, new_lengths = m.draw_windows(c["lengths"])
        assert new_lengths == c["ref_lengths"], name
        for b in range(len(c["lengths"])):
            ids = [A.linspace_round(f, l, n) for f, l, n, _ in windows[owner == b]]
            ids = np.concatenate(ids) if ids else np.zeros(0, dtype=np.int64)
            assert np.array_equal(ids, c["ref_ids"][b, :len(ids)].numpy()), (name, b)
            offs = windows[owner == b][:, 3]
            assert np.array_equal(offs, np.cumsum(windows[owner == b][:, 2]) - windows[owner == b][:, 2])


def test_no_cpu_path():
    from fbkst_b200.augment import SpecAugment, TimeStretch
    b = {"net_input": {"src_tokens": torch.zeros(2, 5, 4), "src_lengths": torch.tensor([5, 3])}}
    with pytest.raises(RuntimeError):
        SpecAugment(2, 2, 1, 1)(b)
    with pytest.raises(RuntimeError):
        TimeStretch(1.0, 2, 0.8, 1.25)(b)
    with pytest.raises(ValueError):
        TimeStretch(1.0, 0, 0.8, 1.25)
