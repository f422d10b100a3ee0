"""Regenerate ``tests/golden/augment.pt`` from the LIVE reference -- TEST INFRASTRUCTURE ONLY.

    python -m oracle.make_golden_augment

Runs the reference's own ``SpecAugment`` (modules/specaugment.py) and ``TimeStretch``
(modules/time_stretch.py) modules on seeded synthetic batches (``random.seed`` / ``np.random.seed``
stored with each case) and keeps inputs and outputs.  Feature 0 of every time-stretch input holds the
frame index, so the reference's index tensors can be read back from its output.  Needs
``/root/reference`` (build container only); the fixture travels, this script's import does not.
"""
import copy
import os
import random

import numpy as np
import torch

from . import golden, ref_loader

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                      "augment.pt")


def batch(seed, lengths, F):
    g = torch.Generator().manual_seed(seed)
    T = max(lengths)
    x = torch.randn(len(lengths), T, F, generator=g) + 3.0  # no exact zeros in the data
    for b, n in enumerate(lengths):
        x[b, n:] = 0
    return x


SPEC_CASES = {
    #        seed lengths                      F   (F_par, T_par, m_F, m_T, rate)
    "default": (11, [120, 97, 64, 30], 40, (13, 13, 2, 2, 1.0)),
    "lb": (12, [300, 280, 150], 40, (27, 100, 1, 1, 1.0)),
    "rate": (13, [80, 80, 70, 60, 50, 40, 30, 20], 24, (15, 70, 2, 2, 0.5)),
    "short": (14, [9, 5], 8, (8, 100, 3, 3, 1.0)),  # T_par > tau, F_par = v
}

STRETCH_CASES = {
    #          seed lengths                 F   (rate, w, low, high)
    "w1": (21, [150, 120, 64, 9], 8, (1.0, 1, 0.8, 1.25)),
    "w5": (22, [203, 150, 77, 12, 7], 40, (1.0, 5, 0.8, 1.25)),
    "w32": (23, [600, 431, 95], 16, (1.0, 32, 0.5, 2.0)),
    "rate": (24, [90, 85, 60, 33, 20, 10], 8, (0.5, 4, 0.8, 1.25)),
    "w100": (25, [1000, 999, 250], 4, (1.0, 100, 0.9, 1.1)),
}


def main():
    ref_loader.load()
    from examples.speech_recognition.modules.specaugment import SpecAugment
    from examples.speech_recognition.modules.time_stretch import TimeStretch

    out = {"spec": {}, "stretch": {}}
    for name, (seed, lengths, F, pars) in SPEC_CASES.items():
        x = batch(seed, lengths, F)
        random.seed(seed); np.random.seed(seed)
        b = {"net_input": {"src_tokens": x.clone(), "src_lengths": torch.tensor(lengths)}}
        y = SpecAugment(*pars)(b)["net_input"]["src_tokens"]
        out["spec"][name] = {"seed": seed, "x": x, "lengths": lengths, "pars": pars, "ref": y.clone()}
        print("spec", name, "zeroed %.3f" % float((y == 0).float().mean()))
    for name, (seed, lengths, F, pars) in STRETCH_CASES.items():
        x = batch(seed, lengths, F)
        x[:, :, 0] = torch.arange(x.shape[1], dtype=torch.float32)[None, :] + 1.0  # frame index + 1
        for b, n in enumerate(lengths):
            x[b, n:] = 0
        random.seed(seed); np.random.seed(seed)
        b = {"net_input": {"src_tokens": x.clone(), "src_lengths": torch.tensor(lengths)}}
        nb = TimeStretch(*pars)(copy.deepcopy(b))
        y, nl = nb["net_input"]["src_tokens"], nb["net_input"]["src_lengths"]
        ids = (y[:, :, 0].round().long() - 1)  # -1 = padding
        out["stretch"][name] = {"seed": seed, "x": x, "lengths": lengths, "pars": pars, "ref": y.clone(),
                                "ref_lengths": nl.tolist(), "ref_ids": ids}
        print("stretch", name, lengths, "->", nl.tolist())
    golden.save(out, GOLDEN)


if __name__ == "__main__":
    main()
