"""Contribution and U'V-product diagnostics on the device (reference: src/utils/diagnostics.py:82-273,528-561 and
compute_uv_correlation_over_time of experiments/multiplicative_strength_comparison.py:46-89).

Same names, arguments and return types as the reference.  The reference materialises the n x n matrices a_i + b_j and
U_i.V_j per time step; libtame_b200 (csrc/tame_align.cu) gets the same sums from r x r Gram matrices computed on the
FP64 tensor cores plus per-time-step row sums -- O(n T r^2) instead of O(n^2 T r).  Undefined values are NaN, as in the
reference: the U'V correlation of a time step where either side's products are all zero (a zero U or V block), and
contributions over no pair (n = 1 with exclude_diagonal).  No CPU implementation: without the CUDA
library these functions raise.  The printing / bookkeeping helpers of the reference module (print_diagnostic_summary,
compare_methods, track_convergence, compute_elbo_gap, compute_reconstruction_error) are host-side utilities outside
the accelerated path and are not provided.
"""
from __future__ import annotations

import ctypes as C
from typing import Tuple

import numpy as np
import torch

from . import _lib
from .alignment import _dev, _prep, _stream


def _contrib_device(X, r, exclude_diagonal):
    """X: (n, T, d) float64 CUDA -> (additive (T,), multiplicative (T,)) float64 CUDA."""
    lib = _lib.load()
    n, T, d = X.shape
    if d != 2 + 2 * r:
        raise ValueError(f"state dimension {d} does not match latent_dim {r} (expected {2 + 2 * r})")
    add = torch.empty(T, dtype=torch.float64, device=X.device)
    mul = torch.empty(T, dtype=torch.float64, device=X.device)
    with torch.cuda.device(X.device):
        _lib.check(lib.tame_contributions(n, T, r, X.data_ptr(), 1 if exclude_diagonal else 0, add.data_ptr(), mul.data_ptr(),
                                          _stream(X.device)))
    return add, mul


def _pad_states(A, M, dev):
    """(n, 2) additive and/or (n, 2r) multiplicative effects -> (n, 1, d) state array with zeros for the missing part."""
    n = (A if A is not None else M).shape[0]
    r = 1 if M is None else M.shape[1] // 2
    a = torch.zeros(n, 2, dtype=torch.float64, device=dev) if A is None else _prep(A, dev)
    m = torch.zeros(n, 2 * r, dtype=torch.float64, device=dev) if M is None else _prep(M, dev)
    return torch.cat([a, m], dim=1).reshape(n, 1, 2 + 2 * r).contiguous(), r


def compute_additive_contribution(A: torch.Tensor, exclude_diagonal: bool = True) -> float:
    """diagnostics.py:82-122: mean over node pairs of (a_i + b_j)^2."""
    X, r = _pad_states(A, None, _dev(A))
    return _contrib_device(X, r, exclude_diagonal)[0].item()


def compute_multiplicative_contribution(M: torch.Tensor, exclude_diagonal: bool = True) -> float:
    """diagnostics.py:125-167: mean over node pairs of (U_i . V_j)^2."""
    X, r = _pad_states(None, M, _dev(M))
    return _contrib_device(X, r, exclude_diagonal)[1].item()


def compute_temporal_contributions(X: torch.Tensor, latent_dim: int, exclude_diagonal: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
    """diagnostics.py:170-217: both contributions at every time step; CPU tensors of shape (T,) in the default dtype
    (the reference fills torch.zeros(T))."""
    add, mul = _contrib_device(_prep(X, _dev(X)), latent_dim, exclude_diagonal)
    dt = torch.get_default_dtype()
    return add.cpu().to(dt), mul.cpu().to(dt)


def compute_contribution_ratio(A: torch.Tensor, M: torch.Tensor) -> float:
    """diagnostics.py:220-251: sqrt(additive / multiplicative), inf when the multiplicative part vanishes."""
    X, r = _pad_states(A, M, _dev(A))
    add, mul = _contrib_device(X, r, True)
    va, vm = add.item(), mul.item()
    if vm < 1e-10:
        return float("inf")
    return np.sqrt(va / vm)


def compute_state_prediction_error(X_true: torch.Tensor, X_pred: torch.Tensor) -> float:
    """diagnostics.py:254-273: mean squared error in state space."""
    lib = _lib.load()
    dev = _dev(X_true)
    a, b = _prep(X_true, dev), _prep(X_pred, dev)
    if a.shape != b.shape:
        a, b = (t.contiguous() for t in torch.broadcast_tensors(a, b))
    out = C.c_double(0.0)
    with torch.cuda.device(dev):
        _lib.check(lib.tame_state_mse(a.numel(), a.data_ptr(), b.data_ptr(), C.byref(out), _stream(dev)))
    return out.value


def compute_uv_correlation_over_time(X_est: torch.Tensor, X_true: torch.Tensor, latent_dim: int) -> torch.Tensor:
    """multiplicative_strength_comparison.py:46-89: correlation of the true and estimated U V' products per time step."""
    lib = _lib.load()
    dev = _dev(X_est)
    e, t = _prep(X_est, dev), _prep(X_true, dev)
    n, T, d = e.shape
    if d != 2 + 2 * latent_dim:
        raise ValueError(f"state dimension {d} does not match latent_dim {latent_dim}")
    corr = torch.empty(T, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.tame_uv_correlation(n, T, latent_dim, e.data_ptr(), t.data_ptr(), corr.data_ptr(), _stream(dev)))
    return corr.cpu().to(torch.get_default_dtype())


def compute_uv_product_correlation(M_est: torch.Tensor, M_true: torch.Tensor, latent_dim: int) -> float:
    """diagnostics.py:528-561: the same for one (n, 2r) pair."""
    dev = _dev(M_est)
    Xe, _ = _pad_states(None, M_est, dev)
    Xt, _ = _pad_states(None, M_true, dev)
    return compute_uv_correlation_over_time(Xe, Xt, latent_dim).double()[0].item()
