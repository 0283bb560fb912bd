"""ORACLE support — the storage format of tests/golden/ref_step_tiny.npz shared by oracle/make_golden.py (writer) and
tests/test_oracle.py (reader).

Step-0 outputs (images, gradients) with more than SKETCH_ABOVE elements are stored as `sketch/<key>` instead of `<key>`,
which keeps the fixture under 1 MB; the initial weights and every smaller array are stored exactly.
"""
import numpy as np
import torch

SKETCH_ABOVE = 2304
SKETCH_K = 64
SKETCH_SEED = 2024


def sketch(t, k=SKETCH_K):
    """k fixed Gaussian projections (float64) of the flattened tensor. For the same projections,
    ||S a - S b|| / ||S b|| estimates ||a - b|| / ||b|| to within about 1 / sqrt(2 k) of its value."""
    a = np.asarray(torch.as_tensor(t).detach().cpu().double()).reshape(-1)
    s = np.random.default_rng([SKETCH_SEED, a.size]).standard_normal((k, a.size))
    return s @ a


def shrink(out):
    """Replace every step-0 array of more than SKETCH_ABOVE elements by its sketch, keeping the order of the others."""
    return {("sketch/" + k if k.startswith("s0/") and v.size > SKETCH_ABOVE else k):
            (sketch(v) if k.startswith("s0/") and v.size > SKETCH_ABOVE else v) for k, v in out.items()}
