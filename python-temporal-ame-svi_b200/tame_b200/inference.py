"""Variational inference for Temporal AME -- host-side mirror of the reference's src/inference/ classes.

Class names, constructor keywords, attributes (`X_mean`, `X_cov`, `n`, `T`, `d`, `r`, `lr`, `history`,
`factorization`), `fit(max_iter, tolerance, verbose, check_every)`, the progress text and the getters are the
reference's (src/inference/base.py:23-343, naive_mf.py:29-396, structured_mf.py:28-338).  What changed is where
the three calls of the fit loop run: `_update_step`, `_compute_elbo` and `_compute_reconstruction_error` are
C-ABI calls into libtame_b200.so (hand-written sm_100a FP64 kernels).  There is no CPU fallback; without a CUDA
device or without the built library these calls raise.

Y is kept on the device in the dtype it arrives in when that is float32 (the reference's default), and widened to FP64
by the kernels as they load it: half the HBM and host->device bytes, the same results bit for bit as a float64 copy
of the same values.  Any other dtype is converted to float64 as before.

Host/device protocol: the variational state lives in HBM while an engine exists; `vi.X_mean` / `vi.X_cov`
are properties that read the device state back on access (and upload on assignment), so reference-style code
that inspects or pickles the object keeps working.  Initialisation stays on the host and issues the reference's
exact sequence of torch RNG calls (structured_mf.py:74-113, naive_mf.py:71-87) so the same seed gives the same
starting point.  The arithmetic is always FP64; tensors are handed back in the dtype the state was created in.
"""
from __future__ import annotations

import ctypes as C
from abc import ABC, abstractmethod
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _lib
from .sharding import DEFAULT_PANEL, owned_rows


def _device_Y(Y: torch.Tensor, dev: torch.device) -> torch.Tensor:
    """Y on `dev` as float32 (kept as it is) or float64 (everything else), contiguous.  A contiguous float32 tensor
    already on `dev` is returned as is: a second copy of the largest Y a GPU holds would not fit next to it."""
    dt = torch.float32 if Y.dtype == torch.float32 else torch.float64
    return Y.detach().to(dev, dt).contiguous()


def _bind_Y(lib, handle, Y: torch.Tensor) -> int:
    """tame_bind_Y or tame_bind_Y_f32, whichever matches Y's dtype (returns the C-ABI code)."""
    return (lib.tame_bind_Y_f32 if Y.dtype == torch.float32 else lib.tame_bind_Y)(handle, Y.data_ptr())


def _fit_config(vi, device_index: int, world: int = 1, rank: int = 0, panel: int = 0):
    """tame_config for a VI object: what the reference reads from `model` inside the loop
    (structured_mf.py:127-128,154-158,177-180,229-237).  Returns (cfg, keepalive arrays)."""
    model = vi.model
    d = vi.d
    f64 = torch.float64
    R = model.R.detach().to("cpu", f64)
    Rinv = model.R_inv.detach().to("cpu", f64)
    S0 = torch.zeros(d, d, dtype=f64)
    S0[:2, :2] = model.Sigma.detach().to("cpu", f64)
    S0[2:, 2:] = model.Psi.detach().to("cpu", f64)
    Q = model.Q.detach().to("cpu", f64)
    keep = [np.ascontiguousarray(model.Phi.detach().to("cpu", f64).numpy()),
            np.ascontiguousarray(torch.linalg.inv(Q).numpy()),          # structured_mf.py:231
            np.ascontiguousarray(torch.linalg.inv(S0).numpy())]         # structured_mf.py:237
    cfg = _lib.TameConfig()
    cfg.n, cfg.T, cfg.r, cfg.mode = vi.n, vi.T, vi.r, vi._mode
    cfg.lr = float(vi.lr)
    for k, v in enumerate(Rinv.reshape(-1).tolist()):
        cfg.Rinv[k] = v
    cfg.logdet_R = float(torch.logdet(R))
    cfg.logdet_Q = float(torch.logdet(Q))
    cfg.logdet_S0 = float(torch.logdet(S0))
    cfg.Phi, cfg.Qinv, cfg.S0inv = (_lib.dptr(a) for a in keep)
    cfg.device, cfg.world, cfg.rank, cfg.panel = device_index, world, rank, panel
    return cfg, keep


class _Engine:
    """Owns one libtame handle plus the device copies of Y (float32 or FP64) / X_mean / X_cov (FP64) as torch CUDA
    tensors."""

    def __init__(self, vi, device=None, world: int = 1, rank: int = 0, panel: int = 0):
        if not torch.cuda.is_available():
            raise RuntimeError("tame_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        model = vi.model
        n, T, r, d = vi.n, vi.T, vi.r, vi.d
        f64 = torch.float64
        cfg, self._keep = _fit_config(vi, dev.index, world, rank, panel)
        self.cfg = cfg
        self.handle = C.c_void_p()
        with torch.cuda.device(dev):
            _lib.check(self.lib.tame_create(C.byref(cfg), C.byref(self.handle)))
            Y = vi.Y if vi.Y is not None else model.Y
            self.Y = _device_Y(Y, dev)
            if tuple(self.Y.shape) != (n, n, T, 2):
                raise ValueError(f"Y has shape {tuple(self.Y.shape)}, expected {(n, n, T, 2)}")
            self.X_mean = torch.empty(n, T, d, dtype=f64, device=dev)
            self.X_cov = torch.empty(n, T, d, d, dtype=f64, device=dev)
            torch.cuda.current_stream(dev).synchronize()
            _lib.check(_bind_Y(self.lib, self.handle, self.Y))
            _lib.check(self.lib.tame_bind_state(self.handle, self.X_mean.data_ptr(), self.X_cov.data_ptr()))
        self._out6 = (C.c_double * 6)()

    def upload(self, X_mean: torch.Tensor, X_cov: torch.Tensor):
        self.X_mean.copy_(X_mean.detach().to(self.device, torch.float64))
        self.X_cov.copy_(X_cov.detach().to(self.device, torch.float64))
        torch.cuda.synchronize(self.device)

    def sweep(self):
        _lib.check(self.lib.tame_sweep(self.handle))

    def elbo_mse(self):
        _lib.check(self.lib.tame_elbo_mse(self.handle, self._out6))
        return list(self._out6)

    def iterate(self):
        _lib.check(self.lib.tame_iterate(self.handle, self._out6))
        return list(self._out6)

    def close(self):
        if self.handle:
            self.lib.tame_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _MultiEngine:
    """One fit sharded over several GPUs of this box, driven from ONE process: a libtame handle per device (rows of Y
    dealt in 64-node panels, X_mean replicated), NCCL for the ELBO all-reduce / the X_cov gather, the fused sweep with
    NVLink peer hand-over (tame_peer_attach).  The ranks' calls are issued from one host thread each (ctypes drops the
    GIL), because every rank's kernels wait for the others'."""

    def __init__(self, vi, devices):
        if not torch.cuda.is_available():
            raise RuntimeError("tame_b200 needs CUDA devices (sm_100a); there is no CPU fallback")
        from concurrent.futures import ThreadPoolExecutor
        self.lib = _lib.load()
        def as_dev(dv):
            if isinstance(dv, int):
                return torch.device("cuda", dv)
            dd = torch.device(dv)
            return torch.device("cuda", dd.index if dd.index is not None else 0)
        self.devs = [as_dev(dv) for dv in devices]
        self.world = len(self.devs)
        if self.world < 2 or self.world > 8 or len({dv.index for dv in self.devs}) != self.world:
            raise ValueError("devices= needs 2..8 distinct CUDA devices")
        n, T, r, d = vi.n, vi.T, vi.r, vi.d
        panel = DEFAULT_PANEL
        if n % panel:
            raise ValueError(f"the multi-GPU fit deals nodes in panels of {panel}: n_nodes={n} must be a multiple of {panel}")
        self.device = self.devs[0]
        self.pool = ThreadPoolExecutor(max_workers=self.world)
        f64 = torch.float64
        Yfull = (vi.Y if vi.Y is not None else vi.model.Y).detach()
        if tuple(Yfull.shape) != (n, n, T, 2):
            raise ValueError(f"Y has shape {tuple(Yfull.shape)}, expected {(n, n, T, 2)}")
        self.rows = [owned_rows(n, panel, self.world, rk) for rk in range(self.world)]
        self.handles, self.Y, self.Xm, self.Xc, self._keep = [], [], [], [], []
        for rk, dv in enumerate(self.devs):
            cfg, keep = _fit_config(vi, dv.index, self.world, rk, panel)
            h = C.c_void_p()
            with torch.cuda.device(dv):
                _lib.check(self.lib.tame_create(C.byref(cfg), C.byref(h)))
                self.Y.append(_device_Y(torch.cat([Yfull[a:b] for a, b in self.rows[rk]], 0), dv))
                self.Xm.append(torch.empty(n, T, d, dtype=f64, device=dv))
                self.Xc.append(torch.empty(n, T, d, d, dtype=f64, device=dv))
                torch.cuda.synchronize(dv)
            self.handles.append(h)
            self._keep.append(keep)
        uid = (C.c_ubyte * 128)()
        _lib.check(self.lib.tame_comm_unique_id(uid))
        self._each(lambda rk: self.lib.tame_comm_init(self.handles[rk], uid))
        table = (C.c_void_p * self.world)(*[h.value for h in self.handles])
        for rk in range(self.world):
            _lib.check(self.lib.tame_peer_attach(self.handles[rk], table))
        self._each(lambda rk: _bind_Y(self.lib, self.handles[rk], self.Y[rk]))
        for rk in range(self.world):
            _lib.check(self.lib.tame_bind_state(self.handles[rk], self.Xm[rk].data_ptr(), self.Xc[rk].data_ptr()))
        self._out6 = [(C.c_double * 6)() for _ in range(self.world)]
        self._gathered = True

    def _each(self, call):
        """call(rank) -> C-ABI return code, on every rank concurrently; the first failure raises."""
        def run(rk):
            with torch.cuda.device(self.devs[rk]):
                return call(rk), (self.lib.tame_last_error() or b"").decode()
        res = list(self.pool.map(run, range(self.world)))
        for rc, msg in res:
            if rc != 0:
                raise RuntimeError(f"libtame_b200: error {rc}: {msg}")

    def upload(self, X_mean: torch.Tensor, X_cov: torch.Tensor):
        for rk, dv in enumerate(self.devs):
            self.Xm[rk].copy_(X_mean.detach().to(dv, torch.float64))
            self.Xc[rk].copy_(X_cov.detach().to(dv, torch.float64))
            torch.cuda.synchronize(dv)

    @property
    def X_mean(self):
        return self.Xm[0]

    @property
    def X_cov(self):
        if not self._gathered:        # X_cov rows of foreign nodes are only valid after the gather
            self._each(lambda rk: self.lib.tame_gather_state(self.handles[rk]))
            self._gathered = True
        return self.Xc[0]

    def sweep(self):
        self._each(lambda rk: self.lib.tame_sweep(self.handles[rk]))
        self._gathered = False

    def elbo_mse(self):
        self._each(lambda rk: self.lib.tame_elbo_mse(self.handles[rk], self._out6[rk]))
        return list(self._out6[0])

    def iterate(self):
        self._each(lambda rk: self.lib.tame_iterate(self.handles[rk], self._out6[rk]))
        self._gathered = False
        return list(self._out6[0])

    def close(self):
        for h in self.handles:
            if h:
                self.lib.tame_destroy(h)
        self.handles = []
        self.pool.shutdown(wait=False)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BaseVariationalInference(ABC):
    """Abstract base of all VI algorithms (base.py:23-272)."""

    def __init__(self, model, learning_rate: float = 0.01, seed: int = 42):
        torch.manual_seed(seed)
        np.random.seed(seed)
        self.model = model
        self.Y = model.Y
        self.n = model.n
        self.lr = learning_rate
        self.history: Dict[str, List[float]] = {"elbo": [], "reconstruction_error": []}
        self._initialize_variational_params()

    @abstractmethod
    def _initialize_variational_params(self) -> None:
        ...

    @abstractmethod
    def _compute_elbo(self) -> float:
        ...

    @abstractmethod
    def _update_step(self) -> None:
        ...

    def fit(self, max_iter: int = 100, tolerance: float = 1e-4, verbose: bool = True,
            check_every: int = 10) -> Dict[str, List[float]]:
        """base.py:127-208: sweep -> ELBO -> MSE per iteration; stop after 3 consecutive iterations whose relative
        ELBO change is below `tolerance`."""
        if verbose:
            print(f"Starting {self.__class__.__name__} optimization...")
            print("=" * 60)
        converged = False
        patience_counter = 0
        prev_elbo = -np.inf
        for iteration in range(max_iter):
            elbo, recon_error = self._iterate()
            self.history["elbo"].append(elbo)
            self.history["reconstruction_error"].append(recon_error)
            if iteration > 0:
                rel_change = abs(elbo - prev_elbo) / (abs(prev_elbo) + 1e-8)
                patience_counter = patience_counter + 1 if rel_change < tolerance else 0
                if patience_counter >= 3:
                    converged = True
            prev_elbo = elbo
            if verbose and (iteration % check_every == 0 or iteration == max_iter - 1):
                self._print_progress(iteration, elbo, recon_error)
            if converged:
                if verbose:
                    print(f"\nConverged at iteration {iteration}")
                break
        if verbose and not converged:
            print("\nReached maximum iterations without convergence")
        return self.history

    def _iterate(self):
        """One body of the fit loop (base.py:171-180)."""
        self._update_step()
        return self._compute_elbo(), self._compute_reconstruction_error()

    def _compute_reconstruction_error(self) -> float:
        if hasattr(self, "get_variational_means"):
            params = self.get_variational_means()
            return self.model.compute_reconstruction_error(*params)
        return 0.0

    def _print_progress(self, iteration: int, elbo: float, recon_error: float) -> None:
        print(f"Iter {iteration:4d} | ELBO: {elbo:10.2f} | MSE: {recon_error:.6f}")

    def get_elbo_history(self) -> List[float]:
        return self.history["elbo"]

    def get_reconstruction_history(self) -> List[float]:
        return self.history["reconstruction_error"]


class BaseTemporalVariationalInference(BaseVariationalInference):
    """Temporal VI base (base.py:275-343) + the device engine shared by the naive and structured classes."""

    _mode = _lib.MODE_GOOD

    def __init__(self, model, learning_rate: float = 0.01, seed: int = 42, device=None, devices=None):
        self.T = model.T
        self.d = model.d
        self.r = model.r
        self._device = device
        self._devices = list(devices) if devices is not None else None      # additive keyword: shard ONE fit over these GPUs
        self._engine: Optional[_Engine] = None
        self._host_mean: Optional[torch.Tensor] = None
        self._host_cov: Optional[torch.Tensor] = None
        self._exact = None             # (X_mean, X_cov) FP64 copies of the device state behind the handed-out tensors
        self._versions = None          # torch in-place version counters of the handed-out tensors at read-back time
        self._device_newer = False     # device state has moved on since the last read-back
        self._host_newer = False       # host tensors were (re)assigned since the last upload
        self._cached = None            # (elbo parts, mse) of the current device state
        super().__init__(model, learning_rate, seed)

    # ---- state: host tensors with lazy device mirroring ------------------------------------------------
    def _pull(self):
        if self._engine is not None and self._device_newer:
            # the device state is FP64; the tensors handed to the caller keep the dtype the state was created in (float32 by
            # default, like the reference).  The exact copy is what a later upload (pickle round trip, resumed fit) uses, unless
            # the caller edited the handed-out tensors in place (their version counters tell).
            m64, c64 = self._engine.X_mean.to("cpu"), self._engine.X_cov.to("cpu")
            self._host_mean = m64.to(self._host_mean.dtype)
            self._host_cov = c64.to(self._host_cov.dtype)
            self._exact = (m64, c64)
            self._versions = (self._host_mean._version, self._host_cov._version)
            self._device_newer = False

    @property
    def X_mean(self) -> torch.Tensor:
        self._pull()
        return self._host_mean

    @X_mean.setter
    def X_mean(self, value: torch.Tensor):
        self._pull()
        self._host_mean = value
        self._host_newer = True
        self._exact = None

    @property
    def X_cov(self) -> torch.Tensor:
        self._pull()
        return self._host_cov

    @X_cov.setter
    def X_cov(self, value: torch.Tensor):
        self._pull()
        self._host_cov = value
        self._host_newer = True
        self._exact = None

    def _ensure_engine(self) -> _Engine:
        if self._engine is None:
            if self.r < 1 or self.r > _lib.MAX_R:
                raise ValueError(f"latent_dim={self.r} is outside the supported range 1..{_lib.MAX_R}")
            self.Y = self.model.Y if self.Y is None else self.Y
            if self._devices is not None and len(self._devices) > 1:
                self._engine = _MultiEngine(self, self._devices)
            else:
                self._engine = _Engine(self, self._devices[0] if self._devices else self._device)
            self._host_newer = True
        edited = (self._versions is not None and not self._device_newer and
                  (self._host_mean._version, self._host_cov._version) != self._versions)     # in-place edit of a handed-out tensor
        if edited:
            self._exact = None
        if self._host_newer or edited:
            if self._exact is not None:
                self._engine.upload(*self._exact)          # bit-exact continuation (unpickled / re-created engine)
            else:
                self._engine.upload(self._host_mean, self._host_cov)
            self._versions = (self._host_mean._version, self._host_cov._version)
            self._host_newer = False
            self._cached = None
        return self._engine

    def __getstate__(self):
        self._pull()
        state = dict(self.__dict__)
        state["_engine"] = None
        state["_device_newer"] = False
        state["_host_newer"] = True
        state["_cached"] = None
        state["_versions"] = None
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)
        if self._host_mean is not None:            # version counters restart with the new tensor objects
            self._versions = (self._host_mean._version, self._host_cov._version)

    # ---- the three calls of the fit loop, on the device -------------------------------------------------
    def _update_step(self) -> None:
        """One Gauss-Seidel sweep (structured_mf.py:211-218 / naive_mf.py:193-205) -> tame_sweep."""
        eng = self._ensure_engine()
        eng.sweep()
        self._device_newer = True
        self._cached = None

    def _elbo_mse(self):
        eng = self._ensure_engine()
        if self._cached is None:
            self._cached = eng.elbo_mse()
        return self._cached

    def _compute_elbo(self) -> float:
        """ELBO of the current state (structured_mf.py:115-122 / naive_mf.py:89-112) -> tame_elbo_mse."""
        return self._elbo_mse()[0]

    def _compute_expected_log_likelihood(self) -> float:
        return self._elbo_mse()[1]

    def _compute_log_prior_initial(self) -> float:
        return self._elbo_mse()[2]

    def _compute_log_prior_transitions(self) -> float:
        return self._elbo_mse()[3]

    def _compute_entropy(self) -> float:
        return self._elbo_mse()[4]

    def _compute_reconstruction_error(self) -> float:
        """base.py:314-326 -> the fused ELBO/MSE kernel's second output."""
        if self._host_mean is None:
            return 0.0
        return self._elbo_mse()[5]

    def _iterate(self):
        eng = self._ensure_engine()
        out = eng.iterate()
        self._device_newer = True
        self._cached = out
        return out[0], out[5]

    def _print_progress(self, iteration: int, elbo: float, recon_error: float) -> None:
        output = f"Iter {iteration:4d} | ELBO: {elbo:10.2f} | MSE: {recon_error:.6f}"
        if hasattr(self, "history") and "state_error" in self.history:
            if len(self.history["state_error"]) > 0:
                output += f" | State MSE: {self.history['state_error'][-1]:.6f}"
        print(output)

    def get_variational_means(self) -> torch.Tensor:
        return self.X_mean

    def get_variational_covariances(self) -> torch.Tensor:
        return self.X_cov


class TemporalAMENaiveMFVI(BaseTemporalVariationalInference):
    """Naive mean-field VI: diagonal block covariances (naive_mf.py:29-396)."""

    _mode = _lib.MODE_NAIVE

    def __init__(self, model, learning_rate: float = 1.0, init_scale: float = 0.1, seed: int = 42, device=None, devices=None):
        self.init_scale = init_scale
        super().__init__(model, learning_rate, seed, device=device, devices=devices)

    def _initialize_variational_params(self) -> None:
        """naive_mf.py:71-87: one randn for the means, 0.5*I covariances."""
        self._host_mean = torch.randn(self.n, self.T, self.d) * self.init_scale
        cov = torch.zeros(self.n, self.T, self.d, self.d)
        cov[:, :] = torch.eye(self.d) * 0.5
        self._host_cov = cov
        self._host_newer = True

    def predict_forward(self, n_steps: int = 1) -> torch.Tensor:
        """naive_mf.py:386-396: iterate the AR(1) map from the last variational mean."""
        X_pred = torch.zeros(self.n, n_steps, self.d)
        Phi = self.model.Phi
        cur = self.X_mean[:, -1].clone()
        for s in range(n_steps):
            cur = torch.matmul(cur, Phi.t())
            X_pred[:, s] = cur
        return X_pred


class TemporalAMEStructuredMFVI(BaseTemporalVariationalInference):
    """Structured mean-field VI, factorization "good" (full d x d blocks) or "bad" ([a,b] independent of [U,V])
    (structured_mf.py:28-338)."""

    def __init__(self, model, factorization: str = "good", learning_rate: float = 1.0, init_scale: float = 0.1,
                 cov_init_scale: float = 0.5, seed: int = 42, device=None, devices=None):
        self.factorization = factorization
        self.init_scale = init_scale
        self.cov_init_scale = cov_init_scale
        self._mode = _lib.MODE_BAD if factorization == "bad" else _lib.MODE_GOOD
        super().__init__(model, learning_rate, seed, device=device, devices=devices)

    def _initialize_variational_params(self) -> None:
        """structured_mf.py:74-113.  The per-block randn calls are kept in the reference's order (means first, then
        one randn(d,d) per block for "good"; randn(2,2) then randn(2r,2r) per block for "bad") because the CPU
        generator's stream depends on the call sizes."""
        n, T, d, r2 = self.n, self.T, self.d, 2 * self.r
        self._host_mean = torch.randn(n, T, d) * self.init_scale
        cov = torch.zeros(n, T, d, d)
        if self.factorization == "good":
            eye = torch.eye(d)
            for i in range(n):
                for t in range(T):
                    blk = eye * self.cov_init_scale + torch.randn(d, d) * 0.01
                    blk = (blk + blk.t()) / 2
                    cov[i, t] = blk + eye * 0.1
        elif self.factorization == "bad":
            e2, e2r = torch.eye(2), torch.eye(r2)
            for i in range(n):
                for t in range(T):
                    top = e2 * self.cov_init_scale + torch.randn(2, 2) * 0.01
                    top = (top + top.t()) / 2 + e2 * 0.05
                    bot = e2r * self.cov_init_scale + torch.randn(r2, r2) * 0.01
                    bot = (bot + bot.t()) / 2 + e2r * 0.05
                    cov[i, t, :2, :2] = top
                    cov[i, t, 2:, 2:] = bot
        else:
            raise ValueError(f"Unknown factorization '{self.factorization}'")
        self._host_cov = cov
        self._host_newer = True

    def get_factorization_type(self) -> str:
        return self.factorization


def fit_batch(vis, max_iter: int = 100, tolerance: float = 1e-4, device=None, n_streams: int = 0, devices=None):
    """Fit many independent VI objects in ONE call (tame_fit_batch; BASELINE config 5, the grid of
    experiments/sensitivity_analysis.py:117-183): every object gets exactly what its own `fit(max_iter, tolerance,
    verbose=False)` would give it -- history appended, state updated, per-fit early stop (base.py:183-203) -- but the
    fits run concurrently on one GPU.  `devices=[0, 1, ...]` deals the fits over several GPUs (independent fits, no
    collective: largest first to the least loaded device), one tame_fit_batch call per device from its own host thread.
    When every object's Y is float32 the fits keep float32 observations on the device (tame_fit_batch_f32); a batch
    with any other dtype widens every Y to float64, which gives the same results.  Returns the list of histories."""
    if not torch.cuda.is_available():
        raise RuntimeError("tame_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    vis = list(vis)
    if not vis:
        return []
    if devices is not None and len(devices) > 1:
        from concurrent.futures import ThreadPoolExecutor
        from .sharding import deal_fits
        groups = deal_fits([float(vi.n) * vi.n * vi.T for vi in vis], len(devices))
        jobs = [(g, d) for g, d in zip(groups, devices) if g]
        with ThreadPoolExecutor(max_workers=len(jobs)) as pool:          # ctypes releases the GIL inside the C call
            futs = [pool.submit(fit_batch, [vis[k] for k in g], max_iter, tolerance, torch.device("cuda", int(d)) if isinstance(d, int) else d, n_streams)
                    for g, d in jobs]
            for fu in futs:
                fu.result()
        return [vi.history for vi in vis]
    if devices is not None and len(devices) == 1 and device is None:
        device = torch.device("cuda", int(devices[0])) if isinstance(devices[0], int) else devices[0]
    lib = _lib.load()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    nf = len(vis)
    f64 = torch.float64
    cfgs = (_lib.TameConfig * nf)()
    Yp, Mp, Cp = (C.c_void_p * nf)(), (C.c_void_p * nf)(), (C.c_void_p * nf)()
    keep = []
    all_f32 = all((vi.Y if vi.Y is not None else vi.model.Y).dtype == torch.float32 for vi in vis)
    ydt = torch.float32 if all_f32 else f64
    for f, vi in enumerate(vis):
        if vi.r < 1 or vi.r > _lib.MAX_R:
            raise ValueError(f"latent_dim={vi.r} is outside the supported range 1..{_lib.MAX_R}")
        vi._pull()
        if vi._engine is not None:            # the batch call works on its own device copies
            vi._engine.close()
            vi._engine = None
        cfg, kk = _fit_config(vi, dev.index)
        Y = (vi.Y if vi.Y is not None else vi.model.Y).detach().to(dev, ydt).contiguous()
        src = vi._exact if (vi._exact is not None and vi._versions == (vi._host_mean._version, vi._host_cov._version)) else (vi._host_mean, vi._host_cov)
        Xm = src[0].detach().to(dev, f64).contiguous()
        Xc = src[1].detach().to(dev, f64).contiguous()
        cfgs[f] = cfg
        Yp[f], Mp[f], Cp[f] = Y.data_ptr(), Xm.data_ptr(), Xc.data_ptr()
        keep.append((kk, Y, Xm, Xc))
    torch.cuda.synchronize(dev)
    el = np.zeros((nf, max(max_iter, 1)))
    ms = np.zeros((nf, max(max_iter, 1)))
    nd = (C.c_int32 * nf)()
    with torch.cuda.device(dev):
        batch = lib.tame_fit_batch_f32 if all_f32 else lib.tame_fit_batch
        _lib.check(batch(nf, cfgs, Yp, Mp, Cp, int(max_iter), float(tolerance), _lib.dptr(el), _lib.dptr(ms), nd, int(n_streams)))
        torch.cuda.synchronize(dev)
    out = []
    for f, vi in enumerate(vis):
        k = int(nd[f])
        vi.history["elbo"].extend(float(x) for x in el[f, :k])
        vi.history["reconstruction_error"].extend(float(x) for x in ms[f, :k])
        m64, c64 = keep[f][2].to("cpu"), keep[f][3].to("cpu")
        vi._host_mean = m64.to(vi._host_mean.dtype)
        vi._host_cov = c64.to(vi._host_cov.dtype)
        vi._exact = (m64, c64)
        vi._versions = (vi._host_mean._version, vi._host_cov._version)
        vi._host_newer = True
        vi._device_newer = False
        vi._cached = None
        out.append(vi.history)
    return out
