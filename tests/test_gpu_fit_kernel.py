"""The whole-fit kernel k_fit (tame_fit_device; every fit of tame_fit_batch's default path, BASELINE config 5) against
the reference's golden vectors and the oracle: every latent dimension, the time-slice widths W = 8 / 16 / 32 of its
ELBO pass and their ragged tails, one / two / four column parts, handles pooled across fits of other shapes, modes and
constants, the device-side stop rule, and Y that is not mirror-consistent.

Every batch asserts its launch count: one k_hab and one k_fit per fit.  A batch that fell back to the host-driven loop
would launch several kernels per iteration and still match the oracle."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, GOLDEN_LONG, METHODS, golden_constants, load_golden, rel_err
from gpu_util import (TOL, UNSTABLE, DeviceFit, make_config, oracle_fit, oracle_pool, random_problem, run_batch,
                      trace_ok)
from oracle import tame_oracle as orc

pytestmark = pytest.mark.gpu
LR = {"naive": 0.3, "good": 0.3, "bad": 0.05}


@pytest.fixture(autouse=True)
def _default_paths(monkeypatch):
    """No inherited switch may move these fits off k_fit or change its team shape / summation order."""
    for v in ("TAME_BATCH", "TAME_SWEEP", "TAME_NH", "TAME_DETERMINISTIC", "TAME_NPARTS", "TAME_BATCH_STREAMS"):
        monkeypatch.delenv(v, raising=False)


def _general_constants(c, rng, R=((0.2, 0.03), (0.03, 0.1))):
    """The constants of `c` with unequal residual variances and a non-diagonal Phi."""
    d = c["d"]
    base = dict(n=c["n"], T=c["T"], r=c["r"], d=d, R=np.array(R), Sigma=c["Sigma"], Psi=c["Psi"],
                Phi=0.7 * np.eye(d) + 0.02 * rng.standard_normal((d, d)), Q=c["Q"])
    return orc.derived_constants(base)


def _check_against(traces, n_done, states, refs):
    for f, ((el, ms), (Gm, Gc), (oel, oms, Om, Oc)) in enumerate(zip(traces, states, refs)):
        assert n_done[f] == len(oel), (f, n_done[f], len(oel))
        assert trace_ok(el, oel), (f, np.max(np.abs(el - oel) / np.abs(oel)))
        assert trace_ok(ms, oms), (f, np.max(np.abs(ms - oms) / np.abs(oms)))
        assert rel_err(Gm, Om) < TOL, (f, rel_err(Gm, Om))
        assert rel_err(Gc, Oc) < TOL, (f, rel_err(Gc, Oc))


# ---- the reference's own numbers ------------------------------------------------------------------------------
@pytest.mark.parametrize("nh", ["default", "1"])
@pytest.mark.parametrize("case", GOLDEN_CASES + GOLDEN_LONG)
def test_golden_through_k_fit(case, nh, monkeypatch):
    """All three methods of a golden case in one batch on ONE stream, so one handle is re-pointed naive -> good -> bad;
    the fixture's own max_iter, tolerance and lr (the 'earlystop' case stops after 50 / 21 / 39 iterations)."""
    if nh == "1":
        monkeypatch.setenv("TAME_NH", "1")
    g = load_golden(case)
    c = golden_constants(g)
    fits = [(c, g["Y"], g[f"{m}_init_mean"], g[f"{m}_init_cov"], float(g["lr"]), orc.MODE_OF[m]) for m in METHODS]
    traces, n_done, states, launches = run_batch(fits, int(g["max_iter"]), float(g["tolerance"]), n_streams=1)
    assert launches == 2 * len(fits)
    for f, m in enumerate(METHODS):
        (el, ms), (Xm, Xc) = traces[f], states[f]
        ref_el, ref_ms = g[f"{m}_elbo"], g[f"{m}_mse"]
        assert n_done[f] == len(ref_el), (m, n_done[f], len(ref_el))
        if (case, m) in UNSTABLE:
            assert trace_ok(el[:2], ref_el[:2], 1e-8) and trace_ok(ms[:2], ref_ms[:2], 1e-8), m
            continue
        assert trace_ok(el, ref_el), (m, np.max(np.abs(el - ref_el) / np.abs(ref_el)))
        assert trace_ok(ms, ref_ms), (m, np.max(np.abs(ms - ref_ms) / np.abs(ref_ms)))
        assert rel_err(Xm, g[f"{m}_final_mean"]) < TOL, m
        assert rel_err(Xc, g[f"{m}_final_cov"]) < TOL, m


# ---- every latent dimension x method, every ELBO slice width, 1 / 2 / 4 column parts ----------------------------
# (r, method) -> (n, T).  T in {1, 2, 7, 16, 32, 33, 64}: slice width W = 8 (T = 1, 2, 7, 33), 16 (T = 16), 32 (T = 32,
# 64), ragged last slices at T = 1, 2, 7, 33; n on both sides of 32 and 64; 200 / 257 nodes: two column parts, 520 / 700:
# four.  r = 4, 5 sum the moment totals in 3 / 2 node parts, r = 6, 7 in one, r = 8 with two entries per thread.
MATRIX = {1: [(520, 1), (12, 64), (33, 7)], 2: [(700, 2), (31, 33), (65, 16)], 3: [(200, 7), (63, 32), (10, 2)],
          4: [(40, 16), (257, 2), (20, 64)], 5: [(64, 7), (33, 32), (520, 2)], 6: [(9, 33), (200, 1), (48, 16)],
          7: [(257, 1), (70, 7), (16, 33)], 8: [(32, 64), (700, 1), (100, 2)]}


def test_matrix_against_oracle():
    """24 fits in one batch; tolerance 0.11 over 8 iterations stops 8 of them early (after 4 or 7 iterations), the
    nearest relative ELBO change sits 1 % from it."""
    max_iter, tol = 8, 0.11
    fits = []
    for r, shapes in MATRIX.items():
        for m, (n, T) in zip(METHODS, shapes):
            c, Y, Xm, Xc = random_problem(n, T, r, seed=500 + 10 * r + n, rho=0.5 if r % 2 else -0.3)
            fits.append((c, Y, Xm, Xc, LR[m], orc.MODE_OF[m]))
    with oracle_pool(len(fits)) as pool:
        jobs = [pool.submit(oracle_fit, Y, Xm, Xc, c, lr, mode, max_iter, tol) for c, Y, Xm, Xc, lr, mode in fits]
        traces, n_done, states, launches = run_batch(fits, max_iter, tol)
        refs = [j.result() for j in jobs]
    assert launches == 2 * len(fits)
    _check_against(traces, n_done, states, refs)
    assert np.sum(n_done < max_iter) >= 4


# ---- BASELINE config 5 at the benchmark's own settings --------------------------------------------------------------
def _config5_problem(n, T, ar, rho, seed):
    """Latents from the model's prior, Y from the device generator (as bench.py's config 5 builds its grid), one
    initial state per method.  Y stays a CUDA tensor shared by the naive and the good fit."""
    from tame_b200 import _lib
    lib = _lib.load()
    r = 2
    c = orc.model_constants(n, T, r, ar_coefficient=ar, rho_dyadic=rho)
    rng = np.random.default_rng(seed)
    L0, Lq = np.linalg.cholesky(c["S0"]), np.linalg.cholesky(c["Q"])
    X = np.zeros((n, T, c["d"]))
    X[:, 0] = rng.standard_normal((n, c["d"])) @ L0.T
    for t in range(1, T):
        X[:, t] = X[:, t - 1] @ c["Phi"].T + rng.standard_normal((n, c["d"])) @ Lq.T
    Xd = torch.as_tensor(X).cuda()
    Y = torch.empty(n, n, T, 2, dtype=torch.float64, device="cuda")
    R = np.ascontiguousarray(c["R"].reshape(4))
    _lib.check(lib.tame_generate_Y(n, T, r, _lib.dptr(R), Xd.data_ptr(), C.c_uint64(seed), 0, n, Y.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    inits = []
    for _ in ("naive", "good"):
        G = rng.standard_normal((n, T, c["d"], c["d"])) * 0.01
        inits.append((rng.standard_normal((n, T, c["d"])) * 0.1, 0.5 * (G + np.swapaxes(G, -1, -2)) + 0.6 * np.eye(c["d"])))
    return c, Y, inits


def test_config5_corners_against_oracle():
    """n in {10, 50, 256} x T in {5, 40} x ar in {0.5, 0.9}, naive + good, r = 2, lr 0.01, tolerance 1e-4 and 150
    iterations as in the benchmark; (256, 40) -- 1.3 s of oracle per iteration -- in a call of its own for 20."""
    lr, tol = 0.01, 1e-4
    groups = {150: [], 20: []}
    for k, (n, T, ar) in enumerate([(n, T, ar) for n in (10, 50, 256) for T in (5, 40) for ar in (0.5, 0.9)]):
        c, Y, inits = _config5_problem(n, T, ar, rho=0.8 if ar == 0.5 else 0.3, seed=900 + k)
        for mode, (Xm, Xc) in zip((orc.NAIVE, orc.GOOD), inits):
            groups[20 if (n, T) == (256, 40) else 150].append((c, Y, Xm, Xc, lr, mode))
    with oracle_pool(sum(len(v) for v in groups.values())) as pool:
        jobs = {it: [pool.submit(oracle_fit, Y.cpu().numpy(), Xm, Xc, c, lr, mode, it, tol) for c, Y, Xm, Xc, lr, mode in fits]
                for it, fits in groups.items()}
        for it, fits in groups.items():
            traces, n_done, states, launches = run_batch(fits, it, tol)
            assert launches == 2 * len(fits)
            _check_against(traces, n_done, states, [j.result() for j in jobs[it]])


# ---- a pooled handle carries nothing from one fit to the next ----------------------------------------------------
# largest n * T first (tame_fit_batch's order): n crosses 192 and 512 and T crosses 32 in both directions between
# neighbours, so one handle (capacity 700 x 50) changes its column-part count and hand-over / H / unit_done layouts
REUSE = [(700, 4), (80, 34), (600, 4), (60, 36), (200, 10), (40, 40), (530, 3), (150, 10), (300, 4), (20, 50), (520, 1),
         (10, 33)]


def test_pooled_handle_reuse_is_invisible(monkeypatch):
    """Under TAME_DETERMINISTIC=1 (fixed summation order) the fits run one after another on one pooled handle give
    bit-identical traces, stop points and states to the same fits each on a fresh handle."""
    monkeypatch.setenv("TAME_DETERMINISTIC", "1")
    assert all(a[0] * a[1] > b[0] * b[1] for a, b in zip(REUSE, REUSE[1:])), "REUSE must be in the batch's run order"
    rng = np.random.default_rng(31)
    fits = []
    for k, (n, T) in enumerate(REUSE):
        c, Y, Xm, Xc = random_problem(n, T, 2, seed=700 + k, rho=(0.6, -0.4, 0.0)[k % 3], ar=(0.9, 0.5, 0.75, 0.6)[k % 4])
        if k % 2:
            c = _general_constants(c, rng, R=((0.1 + 0.02 * k, 0.02), (0.02, 0.1)))
        fits.append((c, Y, Xm, Xc, (0.5, 0.3, 0.05)[k % 3], orc.MODE_OF[METHODS[k % 3]]))
    max_iter, tol = 6, 0.05
    traces, n_done, states, launches = run_batch(fits, max_iter, tol, n_streams=1)
    assert launches == 2 * len(fits)
    for f, fit in enumerate(fits):
        alone_traces, alone_done, alone_states, alone_launches = run_batch([fit], max_iter, tol, n_streams=1)
        assert alone_launches == 2
        assert alone_done[0] == n_done[f], f
        for a, b in zip(alone_traces[0] + alone_states[0], traces[f] + states[f]):
            assert np.array_equal(a, b), (f, np.max(np.abs(a - b)))


# ---- tame_fit_device on a handle of its own -------------------------------------------------------------------------
def _fit_device(fit, max_iter, tol, el_ptr=None):
    """tame_fit_device on a DeviceFit; returns (rc, elbo, mse, n_done) -- traces cut at n_done when rc == 0."""
    el = torch.zeros(max(max_iter, 1), dtype=torch.float64, device="cuda")
    ms = torch.zeros_like(el)
    nd = torch.zeros(1, dtype=torch.int32, device="cuda")
    rc = fit.lib.tame_fit_device(fit.h, max_iter, tol, el.data_ptr() if el_ptr is None else el_ptr, ms.data_ptr(),
                                 nd.data_ptr())
    torch.cuda.synchronize()
    k = int(nd.item())
    return rc, el[:k].cpu().numpy(), ms[:k].cpu().numpy(), k


def _elbo_mse_agree(fit, el, ms):
    """tame_elbo_mse (its own ELBO / MSE kernels) on the state k_fit left: OK (no watchdog abort), and equal to the
    last trace entries -- k_fit's ELBO and MSE are its own code."""
    out = fit.elbo_mse()
    assert abs(out[0] - el[-1]) <= 1e-12 * abs(el[-1]), (out[0], el[-1])
    assert abs(out[5] - ms[-1]) <= 1e-12 * abs(ms[-1]), (out[5], ms[-1])


def test_fit_device_twice_restarts_the_stop_rule():
    """Two calls are two fit()s: the second starts its patience afresh.  Tolerance 1e-3: the first call stops after 8
    of 12 iterations; the second needs 4 (with the first call's patience it would stop after 2)."""
    from tame_b200 import _lib
    c, Y, Xm, Xc = random_problem(72, 9, 3, seed=2024, rho=0.4)
    lr, tol = 0.8, 1e-3
    fit = DeviceFit(Y, Xm, Xc, c, lr, orc.GOOD)
    Om, Oc = Xm.copy(), Xc.copy()
    try:
        for max_iter, expect in ((12, 8), (10, 4)):
            before = fit.lib.tame_launch_count()
            rc, el, ms, k = _fit_device(fit, max_iter, tol)
            _lib.check(rc)
            assert fit.lib.tame_launch_count() - before == 1
            oel, oms = orc.fit(Y, Om, Oc, c, lr, orc.GOOD, max_iter, tol)
            assert k == len(oel) == expect
            assert trace_ok(el, oel) and trace_ok(ms, oms)
            assert rel_err(fit.Xm.cpu().numpy(), Om) < TOL and rel_err(fit.Xc.cpu().numpy(), Oc) < TOL
            _elbo_mse_agree(fit, el, ms)
    finally:
        fit.close()


def test_fit_device_and_sweeps_share_the_epoch():
    """fit_device -> two tame_sweep -> fit_device on one handle equals the oracle: the sweeps' hand-over tags and unit
    stamps continue after the whole-fit kernel's (two column parts at n = 200)."""
    from tame_b200 import _lib
    c, Y, Xm, Xc = random_problem(200, 5, 2, seed=77, rho=0.3)
    lr, mode = 0.5, orc.NAIVE
    fit = DeviceFit(Y, Xm, Xc, c, lr, mode)
    Om, Oc = Xm.copy(), Xc.copy()
    try:
        rc, el, ms, k = _fit_device(fit, 3, 0.0)
        _lib.check(rc)
        oel, oms = orc.fit(Y, Om, Oc, c, lr, mode, 3, 0.0, blocked=True)
        assert k == 3 and trace_ok(el, oel) and trace_ok(ms, oms)
        fit.sweep()
        fit.sweep()
        for _ in range(2):
            orc.sweep_blocked(Y, Om, Oc, c, lr, mode)
        rc, el, ms, k = _fit_device(fit, 3, 0.0)
        _lib.check(rc)
        oel, oms = orc.fit(Y, Om, Oc, c, lr, mode, 3, 0.0, blocked=True)
        assert k == 3 and trace_ok(el, oel) and trace_ok(ms, oms)
        assert rel_err(fit.Xm.cpu().numpy(), Om) < TOL and rel_err(fit.Xc.cpu().numpy(), Oc) < TOL
        _elbo_mse_agree(fit, el, ms)
    finally:
        fit.close()


def test_fit_device_errors(monkeypatch):
    from tame_b200 import _lib
    lib = _lib.load()
    c, Y, Xm, Xc = random_problem(20, 4, 2, seed=3)
    fit = DeviceFit(Y, Xm, Xc, c, 0.3, orc.GOOD)
    try:
        assert _fit_device(fit, 0, 0.0)[0] == -1 and b"max_iter must be positive" in lib.tame_last_error()
        assert _fit_device(fit, 3, 0.0, el_ptr=0)[0] == -1 and b"null argument" in lib.tame_last_error()
        assert np.array_equal(fit.Xm.cpu().numpy(), Xm), "a refused call must not touch the state"
    finally:
        fit.close()
    cfg, keep = make_config(c, 0.3, orc.GOOD)
    h = C.c_void_p()
    _lib.check(lib.tame_create(C.byref(cfg), C.byref(h)))
    try:
        d = torch.zeros(8, dtype=torch.float64, device="cuda")
        assert lib.tame_fit_device(h, 3, 0.0, d.data_ptr(), d.data_ptr(), d.data_ptr()) == -3
        assert b"before tame_bind_Y/tame_bind_state" in lib.tame_last_error()
    finally:
        lib.tame_destroy(h)
    monkeypatch.setenv("TAME_SWEEP", "panel")
    panel = DeviceFit(Y, Xm, Xc, c, 0.3, orc.GOOD)
    try:
        assert _fit_device(panel, 3, 0.0)[0] == -1 and b"needs the single-GPU fused sweep" in lib.tame_last_error()
    finally:
        panel.close()


# ---- Y without the mirror property, general dynamics --------------------------------------------------------------
def test_general_inputs_against_literal_sweep():
    """Y that is not mirror-consistent with a random diagonal (which must be ignored), non-diagonal Phi and unequal
    residual variances, every method, against the oracle's literal node-by-node sweep."""
    rng = np.random.default_rng(8)
    iters, fits = 3, []
    for m, (n, T, r) in zip(METHODS, [(80, 6, 2), (45, 33, 5), (100, 7, 8)]):
        c, Y, Xm, Xc = random_problem(n, T, r, seed=40 + r)
        Y = Y + rng.standard_normal(Y.shape) * 0.3
        Y[np.arange(n), np.arange(n)] = rng.standard_normal((n, T, 2))
        fits.append((_general_constants(c, rng), Y, Xm, Xc, 0.2, orc.MODE_OF[m]))
    traces, n_done, states, launches = run_batch(fits, iters, 0.0)
    assert launches == 2 * len(fits)
    refs = []
    for c, Y, Xm, Xc, lr, mode in fits:
        Om, Oc = Xm.copy(), Xc.copy()
        oel, oms = [], []
        for _ in range(iters):
            orc.sweep(Y, Om, Oc, c, lr, mode)
            oel.append(orc.elbo(Y, Om, Oc, c, mode))
            oms.append(orc.reconstruction_mse(Y, Om, c))
        refs.append((np.array(oel), np.array(oms), Om, Oc))
    _check_against(traces, n_done, states, refs)
