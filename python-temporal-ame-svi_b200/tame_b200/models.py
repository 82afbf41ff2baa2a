"""Generative AME models: the host-side boundary of the hot path.

API mirror of the reference's src/models/{base,static_ame,temporal_ame}.py (class names, constructor keywords,
attribute names, method names).  These classes are plain host code: they hold the hyper-parameters the update
loop reads (R, R_inv, Sigma, Psi, Phi, Q) and produce the synthetic observations.

Same-seed parity: `generate_data()` issues the same sequence of torch RNG draws as the reference
(temporal_ame.py:187-216: one d-vector per node for X^0, one per (node, t>0), then one 2-vector per dyad i<j
per time step, each as `loc + scale_tril @ randn`), so the same constructor arguments under the same torch
default dtype give the same Y.  tests/test_host.py (test_model_mirror_reproduces_reference_data) checks this against the golden fixtures.

Inherited quirk (SURVEY.md fact 5): the reference passes `seed` positionally into the base class's `sigma`
slot (static_ame.py:89 vs base.py:64-74), so the constructor always seeds torch with 42 regardless of
`seed`.  This mirror keeps that behaviour: a drop-in must produce the same data.

`generate_data_device()` is the scalable generator for shapes the O(n^2 T) Python sampling loop cannot reach
(BASELINE configs 3-4): same distribution, Philox stream, written straight into HBM by libtame_b200.
"""
from __future__ import annotations

from abc import ABC, abstractmethod
from typing import Optional, Tuple

import numpy as np
import torch

_BASE_SEED = 42   # what the reference effectively always uses (see module docstring)


def _mvn_factor(cov: torch.Tensor) -> torch.Tensor:
    """scale_tril of torch.distributions.MultivariateNormal(covariance_matrix=cov)."""
    return torch.linalg.cholesky(cov)


def _mvn_draw(loc: torch.Tensor, tril: torch.Tensor) -> torch.Tensor:
    """One MultivariateNormal.sample(): loc + tril @ eps, eps = randn(d) (same RNG consumption)."""
    eps = torch.randn(loc.shape, dtype=loc.dtype)
    return loc + torch.matmul(tril, eps.unsqueeze(-1)).squeeze(-1)


class BaseAMEModel(ABC):
    """Y_ij = [y_ij, y_ji]' ~ N(mu_ij, R), mu_ij = [a_i + b_j + U_i'V_j, a_j + b_i + U_j'V_i]'  (base.py:22-103)."""

    def __init__(self, n_nodes: int, latent_dim: int = 2, sigma: float = 1.0, rho: float = 0.0, seed: int = 42):
        torch.manual_seed(seed)
        np.random.seed(seed)
        self.n = n_nodes
        self.r = latent_dim
        self.sigma = sigma
        self.rho = rho
        s2 = sigma ** 2
        self.R = torch.tensor([[s2, rho * s2], [rho * s2, s2]], dtype=torch.float32)
        self.R_inv = torch.linalg.inv(self.R)
        self.Q = torch.tensor([[0.0, 1.0], [1.0, 0.0]])

    @abstractmethod
    def generate_data(self, **kwargs) -> torch.Tensor:
        ...

    @abstractmethod
    def compute_mean(self, **kwargs) -> torch.Tensor:
        ...

    def _generate_covariance_matrix(self, dim: int, correlation: float = 0.5, variance: float = 1.0) -> torch.Tensor:
        cov = torch.full((dim, dim), 1.0) * correlation * variance
        cov.diagonal().copy_(torch.ones(dim) * variance)
        return cov

    def _block_diagonal_covariance(self, block_sizes, correlations, variances=None) -> torch.Tensor:
        variances = [1.0] * len(block_sizes) if variances is None else variances
        cov = torch.zeros(sum(block_sizes), sum(block_sizes))
        at = 0
        for size, corr, var in zip(block_sizes, correlations, variances):
            cov[at:at + size, at:at + size] = self._generate_covariance_matrix(size, corr, var)
            at += size
        return cov


class StaticAMEModel(BaseAMEModel):
    """Static AME model (static_ame.py:29-324)."""

    def __init__(self, n_nodes: int, latent_dim: int = 2, rho_additive: float = 0.5, rho_multiplicative: float = 0.3,
                 rho_dyadic: float = 0.5, seed: int = 42):
        # the reference forwards `seed` into the base class's `sigma` slot; the RNG seed is therefore always 42
        super().__init__(n_nodes, latent_dim, sigma=seed, rho=0.0, seed=_BASE_SEED)
        self.rho_additive = rho_additive
        self.rho_multiplicative = rho_multiplicative
        self.rho_dyadic = rho_dyadic
        self.R = self._generate_covariance_matrix(dim=2, correlation=rho_dyadic, variance=0.1)
        self.R_inv = torch.linalg.inv(self.R)
        self._initialize_covariances()
        self.A: Optional[torch.Tensor] = None
        self.M: Optional[torch.Tensor] = None
        self.Y: Optional[torch.Tensor] = None

    def _initialize_covariances(self) -> None:
        self.Sigma = self._generate_covariance_matrix(dim=2, correlation=self.rho_additive, variance=1.0)
        self.Psi = self._block_diagonal_covariance([self.r, self.r], [self.rho_multiplicative] * 2, [1.0, 1.0])

    def generate_data(self, return_latents: bool = False):
        tril_A, tril_M, tril_Y = _mvn_factor(self.Sigma), _mvn_factor(self.Psi), _mvn_factor(self.R)
        zero2, zero2r = torch.zeros(2), torch.zeros(2 * self.r)
        self.A = torch.stack([_mvn_draw(zero2, tril_A) for _ in range(self.n)])
        self.M = torch.stack([_mvn_draw(zero2r, tril_M) for _ in range(self.n)])
        mu = self.compute_mean(self.A, self.M)
        self.Y = torch.zeros(self.n, self.n, 2)
        for i in range(self.n):
            for j in range(i + 1, self.n):
                dyad = mu[i, j] + _mvn_draw(zero2, tril_Y)
                self.Y[i, j] = dyad
                self.Y[j, i, 0] = dyad[1]
                self.Y[j, i, 1] = dyad[0]
        if return_latents:
            return self.Y, self.A, self.M
        return self.Y

    def compute_mean(self, A: torch.Tensor, M: torch.Tensor) -> torch.Tensor:
        """mu[i,j] = [a_i + b_j + U_i.V_j, a_j + b_i + U_j.V_i]  (static_ame.py:189-238)."""
        U, V = M[:, :self.r], M[:, self.r:]
        first = (A[:, 0].unsqueeze(1) + A[:, 1].unsqueeze(0)) + torch.matmul(U, V.t())
        return torch.stack([first, first.t()], dim=-1)

    def _offdiag_mean_square(self, field: torch.Tensor) -> float:
        mask = 1 - torch.eye(self.n)
        return (field ** 2 * mask).sum().item() / (self.n * (self.n - 1))

    def compute_reconstruction_error(self, A_est: torch.Tensor, M_est: torch.Tensor) -> float:
        if self.Y is None:
            raise ValueError("No data generated yet. Call generate_data() first.")
        mask = 1 - torch.eye(self.n).unsqueeze(-1)
        err = ((self.Y - self.compute_mean(A_est, M_est)) ** 2) * mask
        return err.sum().item() / (self.n * (self.n - 1))

    def compute_additive_contribution(self, A: torch.Tensor) -> float:
        return self._offdiag_mean_square(A[:, 0].unsqueeze(1) + A[:, 1].unsqueeze(0))

    def compute_multiplicative_contribution(self, M: torch.Tensor) -> float:
        return self._offdiag_mean_square(torch.matmul(M[:, :self.r], M[:, self.r:].t()))


class TemporalAMEModel(StaticAMEModel):
    """Temporal AME model with AR(1) latent dynamics (temporal_ame.py:30-362).

    X_i^t = Phi X_i^{t-1} + eps, eps ~ N(0, Q);  Phi = ar_coefficient * I;
    Q = process_noise_scale * (1 - ar_coefficient^2) * blockdiag(Sigma, Psi).
    """

    def __init__(self, n_nodes: int, n_time: int, latent_dim: int = 2, ar_coefficient: float = 0.8,
                 rho_additive: float = 0.5, rho_multiplicative: float = 0.3, rho_dyadic: float = 0.5,
                 process_noise_scale: float = 0.1, seed: int = 42):
        super().__init__(n_nodes=n_nodes, latent_dim=latent_dim, rho_additive=rho_additive,
                         rho_multiplicative=rho_multiplicative, rho_dyadic=rho_dyadic, seed=seed)
        self.r = latent_dim
        self.T = n_time
        self.ar_coefficient = ar_coefficient
        self.process_noise_scale = process_noise_scale
        self.d = 2 + 2 * self.r
        self._initialize_dynamics()
        self.X: Optional[torch.Tensor] = None
        self.Y: Optional[torch.Tensor] = None

    def _stationary_cov(self) -> torch.Tensor:
        s = torch.zeros(self.d, self.d)
        s[:2, :2] = self.Sigma
        s[2:, 2:] = self.Psi
        return s

    def _initialize_dynamics(self) -> None:
        self.Phi = torch.eye(self.d) * self.ar_coefficient
        self.Q = (1 - self.ar_coefficient ** 2) * self._stationary_cov()
        self.Q = self.Q * self.process_noise_scale

    def generate_data(self, return_latents: bool = False):
        """Host generator with the reference's RNG stream (temporal_ame.py:147-220)."""
        n, T, d = self.n, self.T, self.d
        self.X = torch.zeros(n, T, d)
        self.Y = torch.zeros(n, n, T, 2)
        tril0, trilq, trilr = _mvn_factor(self._stationary_cov()), _mvn_factor(self.Q), _mvn_factor(self.R)
        zd, z2 = torch.zeros(d), torch.zeros(2)
        for i in range(n):
            self.X[i, 0] = _mvn_draw(zd, tril0)
            for t in range(1, T):
                self.X[i, t] = torch.matmul(self.Phi, self.X[i, t - 1]) + _mvn_draw(zd, trilq)
        for t in range(T):
            mu_t = self.compute_mean(self.X[:, t, :2], self.X[:, t, 2:])
            for i in range(n):
                for j in range(i + 1, n):
                    dyad = mu_t[i, j] + _mvn_draw(z2, trilr)
                    self.Y[i, j, t] = dyad
                    self.Y[j, i, t, 0] = dyad[1]
                    self.Y[j, i, t, 1] = dyad[0]
        if return_latents:
            return self.Y, self.X
        return self.Y

    def generate_latents_fast(self, seed: int = 42) -> torch.Tensor:
        """Vectorised AR(1) latent trajectories in float64 (same distribution as generate_data, not the same
        stream): one batched draw per time step.  Used with generate_data_device for large shapes."""
        g = torch.Generator().manual_seed(seed)
        n, T, d = self.n, self.T, self.d
        tril0 = _mvn_factor(self._stationary_cov().double())
        trilq = _mvn_factor(self.Q.double())
        Phi = self.Phi.double()
        X = torch.zeros(n, T, d, dtype=torch.float64)
        X[:, 0] = torch.randn(n, d, generator=g, dtype=torch.float64) @ tril0.T
        for t in range(1, T):
            X[:, t] = X[:, t - 1] @ Phi.T + torch.randn(n, d, generator=g, dtype=torch.float64) @ trilq.T
        return X

    def generate_data_device(self, device="cuda", seed: int = 42, row_begin: int = 0, row_end: Optional[int] = None,
                             keep_on_device: bool = True, dtype: torch.dtype = torch.float64):
        """Scalable generator: latents on the host (O(nTd)), observations written directly into HBM by the
        tame_generate_Y kernel (same distribution as temporal_ame.py:200-216, Philox keyed by (dyad, t)).
        Returns rows [row_begin, row_end) of Y as a CUDA tensor of `dtype`; `self.Y` is set to it (full rows only).
        dtype=torch.float32 computes in float64 and rounds once per value (tame_generate_Y_f32): half the HBM, and
        the fits keep it as float32 on the device.  Other dtypes raise ValueError."""
        import ctypes as C
        from . import _lib
        if dtype not in (torch.float64, torch.float32):
            raise ValueError(f"generate_data_device: dtype must be torch.float64 or torch.float32, not {dtype}")
        lib = _lib.load()
        gen = lib.tame_generate_Y_f32 if dtype == torch.float32 else lib.tame_generate_Y
        row_end = self.n if row_end is None else row_end
        dev = torch.device(device)
        self.X = self.generate_latents_fast(seed)
        Xd = self.X.to(dev)
        Y = torch.empty(row_end - row_begin, self.n, self.T, 2, dtype=dtype, device=dev)
        R = np.ascontiguousarray(self.R.double().numpy().reshape(4))
        with torch.cuda.device(dev):
            _lib.check(gen(self.n, self.T, self.r, _lib.dptr(R), Xd.data_ptr(), C.c_uint64(seed),
                                           row_begin, row_end, Y.data_ptr(),
                                           torch.cuda.current_stream(dev).cuda_stream))
            torch.cuda.synchronize(dev)
        if row_begin == 0 and row_end == self.n:
            self.Y = Y if keep_on_device else Y.cpu()
        return Y

    def get_states_at_time(self, t: int) -> Tuple[torch.Tensor, torch.Tensor]:
        if self.X is None:
            raise ValueError("No data generated yet. Call generate_data() first.")
        if t < 0 or t >= self.T:
            raise ValueError(f"Time index {t} out of bounds [0, {self.T}).")
        return self.X[:, t, :2], self.X[:, t, 2:]

    def compute_temporal_reconstruction_error(self, X_est: torch.Tensor) -> float:
        """Host version of the reconstruction MSE (temporal_ame.py:255-291).  The VI classes use the fused CUDA
        kernel instead; this stays for API compatibility."""
        if self.Y is None:
            raise ValueError("No data generated yet. Call generate_data() first.")
        Y = self.Y.to(X_est.device) if self.Y.device != X_est.device else self.Y
        mask = 1 - torch.eye(self.n, device=X_est.device).unsqueeze(-1)
        total = 0.0
        for t in range(self.T):
            mu = self.compute_mean(X_est[:, t, :2], X_est[:, t, 2:])
            total += (((Y[:, :, t] - mu) ** 2) * mask).sum().item()
        return total / (self.n * (self.n - 1) * self.T)

    def compute_state_prediction_error(self, X_est: torch.Tensor) -> float:
        if self.X is None:
            raise ValueError("No data generated yet. Call generate_data() first.")
        return ((self.X - X_est) ** 2).mean().item()

    def compute_temporal_additive_contribution(self, X: torch.Tensor) -> torch.Tensor:
        out = torch.zeros(self.T)
        for t in range(self.T):
            out[t] = self.compute_additive_contribution(X[:, t, :2])
        return out

    def compute_temporal_multiplicative_contribution(self, X: torch.Tensor) -> torch.Tensor:
        out = torch.zeros(self.T)
        for t in range(self.T):
            out[t] = self.compute_multiplicative_contribution(X[:, t, 2:])
        return out
