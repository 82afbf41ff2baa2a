"""Shared test plumbing: marker registration, import paths, golden-fixture loader."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "python-temporal-ame-svi_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
GOLDEN_CASES = ["conftest_lr1", "conftest_lr001", "r3_rho08", "r1_T1", "r4_T2", "earlystop", "config1", "config2"]
GOLDEN_LONG = ["config2_long"]       # BASELINE config 2, 50 iterations of every method (too slow for the literal-oracle loop)
METHODS = ["naive", "good", "bad"]


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def load_golden(name):
    path = os.path.join(GOLDEN_DIR, name + ".npz")
    if not os.path.exists(path):
        pytest.skip(f"golden fixture {name}.npz not generated")
    z = np.load(path)
    g = {k: z[k] for k in z.files}
    if "inputs" in g:           # runs of one problem share its inputs (Y, X_true, initial states) in one fixture
        g = {**load_golden(str(g.pop("inputs"))), **g}
    if "Y0" in g:               # mirror-consistent Y stored as its first channel: Y[i, j, t, 1] == Y[j, i, t, 0]
        Y0 = g.pop("Y0")
        g["Y"] = np.stack([Y0, np.swapaxes(Y0, 0, 1)], axis=-1)
    return g


def golden_constants(g):
    """Oracle constants dict from the hyper-parameters stored in a golden fixture."""
    from oracle import tame_oracle as orc
    n, T, r = int(g["n"]), int(g["T"]), int(g["r"])
    return orc.derived_constants(dict(n=n, T=T, r=r, d=2 + 2 * r, R=g["R"], R_inv=g["R_inv"], Sigma=g["Sigma"],
                                      Psi=g["Psi"], Phi=g["Phi"], Q=g["Q"]))


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-300))
