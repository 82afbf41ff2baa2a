"""Helpers for the -m gpu tests: call libtame_b200 through its C ABI with numpy buffers, seeded problems, and the
oracle's fit in worker processes."""
import ctypes as C
import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor

import numpy as np

from oracle import tame_oracle as orc

TOL = 1e-9
# divergent iterations in the reference itself ('bad' with a large step): rounding differences are amplified
# each sweep, so the comparison window is the first iterations and the tolerance widens with the sweep count.
UNSTABLE = {("conftest_lr1", "bad"), ("r3_rho08", "bad"), ("r1_T1", "bad"), ("r4_T2", "bad")}


def trace_ok(a, b, tol=TOL):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.all(np.abs(a - b) <= tol * np.abs(b))


def random_problem(n, T, r, seed, rho=0.5, ar=0.8):
    """Mirror-consistent Y with zero diagonal from seeded latents, and a perturbed 'good'-style initial state."""
    rng = np.random.default_rng(seed)
    c = orc.model_constants(n, T, r, ar_coefficient=ar, rho_dyadic=rho)
    d = c["d"]
    X = rng.standard_normal((n, T, d)) * 0.7
    Y = np.zeros((n, n, T, 2))
    Lr = np.linalg.cholesky(c["R"])
    for t in range(T):
        mu = orc.compute_mean(X[:, t, :2], X[:, t, 2:], r)
        eps = rng.standard_normal((n, n, 2)) @ Lr.T
        yt = mu + eps
        iu = np.triu_indices(n, 1)
        Y[iu[0], iu[1], t] = yt[iu]
        Y[iu[1], iu[0], t, 0] = yt[iu][:, 1]
        Y[iu[1], iu[0], t, 1] = yt[iu][:, 0]
    Xm = rng.standard_normal((n, T, d)) * 0.1
    G = rng.standard_normal((n, T, d, d)) * 0.01
    Xc = 0.6 * np.eye(d) + 0.5 * (G + np.swapaxes(G, -1, -2))
    return c, Y, Xm, Xc


def make_config(c, lr, mode, device=0, world=1, rank=0, panel=0):
    """tame_config from an oracle constants dict.  Returns (cfg, keepalive)."""
    from tame_b200 import _lib
    cfg = _lib.TameConfig()
    cfg.n, cfg.T, cfg.r, cfg.mode = int(c["n"]), int(c["T"]), int(c["r"]), int(mode)
    cfg.lr = float(lr)
    for k, v in enumerate(np.asarray(c["R_inv"], dtype=np.float64).reshape(-1)):
        cfg.Rinv[k] = float(v)
    cfg.logdet_R, cfg.logdet_Q, cfg.logdet_S0 = float(c["logdet_R"]), float(c["logdet_Q"]), float(c["logdet_S0"])
    keep = [np.ascontiguousarray(c[k], dtype=np.float64) for k in ("Phi", "Q_inv", "S0_inv")]
    cfg.Phi, cfg.Qinv, cfg.S0inv = (_lib.dptr(a) for a in keep)
    cfg.device, cfg.world, cfg.rank, cfg.panel = device, world, rank, panel
    return cfg, keep


def fit_host(Y, Xm, Xc, c, lr, mode, max_iter, tol=0.0):
    """tame_fit_host on copies of the inputs; returns (elbo_trace, mse_trace, Xm, Xc)."""
    from tame_b200 import _lib
    lib = _lib.load()
    cfg, keep = make_config(c, lr, mode)
    Y = np.ascontiguousarray(Y, dtype=np.float64)
    Xm = np.ascontiguousarray(Xm, dtype=np.float64).copy()
    Xc = np.ascontiguousarray(Xc, dtype=np.float64).copy()
    el = np.zeros(max(max_iter, 1))
    ms = np.zeros(max(max_iter, 1))
    nd = C.c_int32(0)
    _lib.check(lib.tame_fit_host(C.byref(cfg), Y.ctypes.data, Xm.ctypes.data, Xc.ctypes.data, max_iter, float(tol),
                                 _lib.dptr(el), _lib.dptr(ms), C.byref(nd)))
    return el[:nd.value], ms[:nd.value], Xm, Xc


class DeviceFit:
    """Handle-level access (tame_create / bind / sweep / elbo_mse) with torch CUDA tensors as storage."""

    def __init__(self, Y, Xm, Xc, c, lr, mode, device=0):
        import torch
        from tame_b200 import _lib
        self._lib_mod = _lib
        self.lib = _lib.load()
        self.cfg, self._keep = make_config(c, lr, mode, device=device)
        dev = torch.device("cuda", device)
        self.Y = torch.as_tensor(np.ascontiguousarray(Y), dtype=torch.float64).to(dev) if not hasattr(Y, "data_ptr") else Y
        self.Xm = torch.as_tensor(np.ascontiguousarray(Xm), dtype=torch.float64).to(dev) if not hasattr(Xm, "data_ptr") else Xm
        self.Xc = torch.as_tensor(np.ascontiguousarray(Xc), dtype=torch.float64).to(dev) if not hasattr(Xc, "data_ptr") else Xc
        torch.cuda.synchronize(dev)
        self.h = C.c_void_p()
        _lib.check(self.lib.tame_create(C.byref(self.cfg), C.byref(self.h)))
        _lib.check(self.lib.tame_bind_Y(self.h, self.Y.data_ptr()))
        _lib.check(self.lib.tame_bind_state(self.h, self.Xm.data_ptr(), self.Xc.data_ptr()))
        self.out = (C.c_double * 6)()

    def sweep(self):
        self._lib_mod.check(self.lib.tame_sweep(self.h))

    def elbo_mse(self):
        self._lib_mod.check(self.lib.tame_elbo_mse(self.h, self.out))
        return np.array(list(self.out))

    def close(self):
        if self.h:
            self.lib.tame_destroy(self.h)
            self.h = C.c_void_p()


class DeviceFit32(DeviceFit):
    """DeviceFit with Y stored as float32 (a float32 CUDA tensor is used in place) and bound with tame_bind_Y_f32"""

    def __init__(self, Y, Xm, Xc, c, lr, mode, device=0):
        import torch
        from tame_b200 import _lib
        self._lib_mod = _lib
        self.lib = _lib.load()
        self.cfg, self._keep = make_config(c, lr, mode, device=device)
        dev = torch.device("cuda", device)
        self.Y = torch.as_tensor(np.ascontiguousarray(Y, dtype=np.float32)).to(dev) if not hasattr(Y, "data_ptr") else Y
        self.Xm = torch.as_tensor(np.ascontiguousarray(Xm), dtype=torch.float64).to(dev) if not hasattr(Xm, "data_ptr") else Xm
        self.Xc = torch.as_tensor(np.ascontiguousarray(Xc), dtype=torch.float64).to(dev) if not hasattr(Xc, "data_ptr") else Xc
        torch.cuda.synchronize(dev)
        self.h = C.c_void_p()
        _lib.check(self.lib.tame_create(C.byref(self.cfg), C.byref(self.h)))
        _lib.check(self.lib.tame_bind_Y_f32(self.h, self.Y.data_ptr()))
        _lib.check(self.lib.tame_bind_state(self.h, self.Xm.data_ptr(), self.Xc.data_ptr()))
        self.out = (C.c_double * 6)()


def run_batch(fits, max_iter, tol, n_streams=0):
    """tame_fit_batch over `fits` = [(c, Y, Xm, Xc, lr, mode), ...] on fresh device copies of the state (Y may be a CUDA
    tensor already, shared by several fits).  Returns (traces, n_done, states, launches): traces[f] = (elbo, mse) cut at
    n_done[f], states[f] = (X_mean, X_cov) after the fit, launches = kernels the call launched (tame_launch_count)."""
    import torch
    from tame_b200 import _lib
    lib = _lib.load()
    nf = len(fits)
    cfgs = (_lib.TameConfig * nf)()
    Yp, Mp, Cp = (C.c_void_p * nf)(), (C.c_void_p * nf)(), (C.c_void_p * nf)()
    keep, dev = [], []
    for f, (c, Y, Xm, Xc, lr, mode) in enumerate(fits):
        cfgs[f], kk = make_config(c, lr, mode)
        keep.append(kk)
        Yd = Y if isinstance(Y, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(Y), dtype=torch.float64).cuda()
        t = [Yd] + [torch.as_tensor(np.array(a, dtype=np.float64)).cuda() for a in (Xm, Xc)]
        dev.append(t)
        Yp[f], Mp[f], Cp[f] = t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr()
    torch.cuda.synchronize()
    el, ms, nd = np.zeros((nf, max_iter)), np.zeros((nf, max_iter)), (C.c_int32 * nf)()
    before = lib.tame_launch_count()
    _lib.check(lib.tame_fit_batch(nf, cfgs, Yp, Mp, Cp, max_iter, tol, _lib.dptr(el), _lib.dptr(ms), nd, n_streams))
    launches = lib.tame_launch_count() - before
    n_done = np.array(list(nd))
    traces = [(el[f, :n_done[f]], ms[f, :n_done[f]]) for f in range(nf)]
    states = [(t[1].cpu().numpy(), t[2].cpu().numpy()) for t in dev]
    return traces, n_done, states, launches


def oracle_fit(Y, Xm, Xc, c, lr, mode, max_iter, tol):
    """orc.fit on copies of the state (blocked schedule above 80 nodes); returns (elbo, mse, X_mean, X_cov)."""
    Xm, Xc = np.array(Xm, dtype=np.float64), np.array(Xc, dtype=np.float64)
    el, ms = orc.fit(Y, Xm, Xc, c, lr, mode, max_iter, tol, blocked=c["n"] > 80)
    return el, ms, Xm, Xc


def oracle_pool(n_jobs):
    """Worker processes for oracle_fit: the oracle is a serial Python loop over (node, time) cells and independent fits
    are independent, so a batch of them is checked in the time of its longest fit on a machine with enough cores.
    'spawn': the workers never inherit the parent's CUDA context."""
    workers = max(1, min(n_jobs, len(os.sched_getaffinity(0))))
    return ProcessPoolExecutor(workers, mp_context=multiprocessing.get_context("spawn"))
