"""Loader of the BNN-training fixtures (tests/golden/train_*.npz, written by oracle/make_golden_train.py).

A fixture may keep some of its arrays in `<tag>.<name>.npz` beside `<tag>.npz` (the recorded dropout noise of a
large network), so that no single file passes 1 MB; `load` merges the parts."""
import glob
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def train_tags():
    return sorted(t for t in (os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "train_*.npz")))
                  if "." not in t)


def load(tag):
    fx = {}
    for path in [os.path.join(GOLDEN_DIR, tag + ".npz")] + sorted(glob.glob(os.path.join(GOLDEN_DIR, tag + ".*.npz"))):
        raw = np.load(path)
        fx.update({k: (torch.from_numpy(np.array(raw[k])) if raw[k].ndim else raw[k].item()) for k in raw.files})
    fx["dtype"] = fx["X"].dtype
    return fx


def augmented_inputs(fx):
    """[x_nonang, sin, cos, u] of the cartpole dataset (angle index 2), as fit() forms it (modules.py:158-163)."""
    X, U = fx["X"], fx["U"]
    return torch.cat([X[:, [0, 1, 3]], X[:, 2:3].sin(), X[:, 2:3].cos(), U], -1)
