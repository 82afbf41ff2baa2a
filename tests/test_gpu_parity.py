"""Parity of the CUDA path (through the C ABI / the drop-in classes) with the golden vectors of the reference
and with the oracle.  Tolerance: rel 1e-9 on means, covariances, ELBO trace and MSE trace (north_star)."""
import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, GOLDEN_LONG, METHODS, golden_constants, load_golden, rel_err
from gpu_util import TOL, UNSTABLE, random_problem, trace_ok
from oracle import tame_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _float64_default():
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    yield
    torch.set_default_dtype(old)


@pytest.mark.parametrize("meth", METHODS)
@pytest.mark.parametrize("case", GOLDEN_CASES + GOLDEN_LONG)
def test_c_abi_fit_matches_reference_golden(case, meth):
    """tame_fit_host (host buffers in, host buffers out) on the reference's own Y and initial state."""
    from gpu_util import fit_host
    g = load_golden(case)
    c = golden_constants(g)
    el, ms, Xm, Xc = fit_host(g["Y"], g[f"{meth}_init_mean"], g[f"{meth}_init_cov"], c, float(g["lr"]),
                              orc.MODE_OF[meth], int(g["max_iter"]), float(g["tolerance"]))
    ref_el, ref_ms = g[f"{meth}_elbo"], g[f"{meth}_mse"]
    assert len(el) == len(ref_el), "early-stop iteration differs"
    if (case, meth) in UNSTABLE:
        assert trace_ok(el[:2], ref_el[:2], 1e-8) and trace_ok(ms[:2], ref_ms[:2], 1e-8)
        return
    assert trace_ok(el, ref_el), np.max(np.abs(el - ref_el) / np.abs(ref_el))
    assert trace_ok(ms, ref_ms), np.max(np.abs(ms - ref_ms) / np.abs(ref_ms))
    assert rel_err(Xm, g[f"{meth}_final_mean"]) < TOL
    assert rel_err(Xc, g[f"{meth}_final_cov"]) < TOL


@pytest.mark.parametrize("meth", METHODS)
@pytest.mark.parametrize("case", ["conftest_lr001", "config1"])
def test_drop_in_classes_match_reference_golden(case, meth):
    """The reference's own call sequence: model -> generate_data -> VI(model) -> fit -> history / X_mean / X_cov."""
    from src.models import TemporalAMEModel
    from src.inference import TemporalAMENaiveMFVI, TemporalAMEStructuredMFVI
    g = load_golden(case)
    model = TemporalAMEModel(**eval(str(g["model_kwargs"])))
    model.generate_data()
    lr = float(g["lr"])
    vi = (TemporalAMENaiveMFVI(model, learning_rate=lr, seed=42) if meth == "naive"
          else TemporalAMEStructuredMFVI(model, factorization=meth, learning_rate=lr, seed=42))
    iters = min(int(g["max_iter"]), 25)
    hist = vi.fit(max_iter=iters, tolerance=0.0, verbose=False)
    assert hist is vi.history and len(hist["elbo"]) == iters
    assert trace_ok(hist["elbo"], g[f"{meth}_elbo"][:iters])
    assert trace_ok(hist["reconstruction_error"], g[f"{meth}_mse"][:iters])
    if iters == int(g["max_iter"]):
        assert rel_err(vi.get_variational_means().numpy(), g[f"{meth}_final_mean"]) < TOL
        assert rel_err(vi.get_variational_covariances().numpy(), g[f"{meth}_final_cov"]) < TOL
        parts = [vi._compute_expected_log_likelihood(), vi._compute_log_prior_initial(),
                 vi._compute_log_prior_transitions(), vi._compute_entropy()]
        assert trace_ok(parts, g[f"{meth}_parts"])
    # a second fit() continues from the current state and appends to the same history (base.py:176-180)
    vi.fit(max_iter=2, tolerance=0.0, verbose=False)
    assert len(vi.history["elbo"]) == iters + 2


# shapes that cross the 64-node block boundary (upper pass, pushes, several chain launches), ragged n and T,
# every supported latent dimension, T above one warp-slice
SHAPES = [(70, 3, 1), (65, 7, 2), (130, 5, 3), (96, 33, 4), (64, 4, 5), (100, 2, 6), (67, 9, 7), (129, 6, 8), (200, 40, 2)]


@pytest.fixture(params=["fused", "fused-nh1", "panel"])
def sweep_path(request, monkeypatch):
    """The schedulers of the same sweep: the persistent fused kernel in both team shapes (chain + totals + two input warps
    per time step -- the default at these sizes -- and chain + one helper, TAME_NH=1) and the stream-ordered per-panel
    launches (the multi-GPU fallback, forced here on one GPU)."""
    monkeypatch.delenv("TAME_SWEEP", raising=False)
    monkeypatch.delenv("TAME_NH", raising=False)
    if request.param == "panel":
        monkeypatch.setenv("TAME_SWEEP", "panel")
    elif request.param == "fused-nh1":
        monkeypatch.setenv("TAME_NH", "1")
    return request.param


@pytest.mark.parametrize("meth", METHODS)
@pytest.mark.parametrize("shape", SHAPES)
def test_c_abi_matches_oracle_on_seeded_inputs(shape, meth, sweep_path):
    from gpu_util import fit_host
    n, T, r = shape
    c, Y, Xm, Xc = random_problem(n, T, r, seed=1000 + n + T + r, rho=0.5 if r % 2 else -0.3)
    lr = 0.05 if meth == "bad" else 0.3
    mode = orc.MODE_OF[meth]
    iters = 2
    el, ms, Gm, Gc = fit_host(Y, Xm, Xc, c, lr, mode, iters)
    Om, Oc = Xm.copy(), Xc.copy()
    oel, oms = [], []
    for _ in range(iters):
        orc.sweep_fast(Y, Om, Oc, c, lr, mode)
        oel.append(orc.elbo(Y, Om, Oc, c, mode))
        oms.append(orc.reconstruction_mse(Y, Om, c))
    assert rel_err(Gm, Om) < TOL, rel_err(Gm, Om)
    assert rel_err(Gc, Oc) < TOL, rel_err(Gc, Oc)
    assert trace_ok(el, oel) and trace_ok(ms, oms)


def test_asymmetric_Y_and_general_dynamics():
    """Y that is NOT mirror-consistent (experiments/multiplicative_strength_comparison.py:168-185 overrides
    model.Y by hand) and a non-diagonal Phi: nothing in the kernels may assume Y[j,i,t,0] == Y[i,j,t,1]."""
    from gpu_util import fit_host
    rng = np.random.default_rng(7)
    n, T, r = 80, 6, 2
    c, Y, Xm, Xc = random_problem(n, T, r, seed=5)
    Y = Y + rng.standard_normal(Y.shape) * 0.3
    Y[np.arange(n), np.arange(n)] = rng.standard_normal((n, T, 2))     # diagonal must be ignored
    d = c["d"]
    base = dict(n=n, T=T, r=r, d=d, R=np.array([[0.2, 0.03], [0.03, 0.1]]), Sigma=c["Sigma"], Psi=c["Psi"],
                Phi=0.7 * np.eye(d) + 0.02 * rng.standard_normal((d, d)), Q=c["Q"])
    c2 = orc.derived_constants(base)
    for meth in METHODS:
        mode = orc.MODE_OF[meth]
        el, ms, Gm, Gc = fit_host(Y, Xm, Xc, c2, 0.2, mode, 2)
        Om, Oc = Xm.copy(), Xc.copy()
        for _ in range(2):
            orc.sweep(Y, Om, Oc, c2, 0.2, mode)
        assert rel_err(Gm, Om) < TOL and rel_err(Gc, Oc) < TOL
        assert abs(el[-1] - orc.elbo(Y, Om, Oc, c2, mode)) <= TOL * abs(el[-1])
        assert abs(ms[-1] - orc.reconstruction_mse(Y, Om, c2)) <= TOL * abs(ms[-1])


def test_handle_level_calls_and_properties():
    """tame_sweep / tame_elbo_mse on device buffers; ELBO parts add up; a sweep with lr=0 is the identity;
    'bad' keeps its cross blocks at zero; naive covariances stay diagonal (test_inference.py:187-203, 37-43)."""
    from gpu_util import DeviceFit
    n, T, r = 90, 5, 2
    c, Y, Xm, Xc = random_problem(n, T, r, seed=11)
    f = DeviceFit(Y, Xm, Xc, c, 0.0, orc.GOOD)
    before = f.elbo_mse()
    f.sweep()
    torch.cuda.synchronize()
    assert np.array_equal(f.Xm.cpu().numpy(), Xm) and np.array_equal(f.Xc.cpu().numpy(), Xc)
    after = f.elbo_mse()
    assert np.array_equal(before, after)
    assert abs(before[0] - before[1:5].sum()) <= 1e-12 * abs(before[0])
    parts = orc.elbo_parts(Y, Xm, Xc, c, orc.GOOD)
    assert np.all(np.abs(before[1:5] - np.array(parts)) <= TOL * np.abs(np.array(parts)))
    f.close()
    fb = DeviceFit(Y, Xm, Xc, c, 1.0, orc.BAD)
    fb.sweep()
    torch.cuda.synchronize()
    cov = fb.Xc.cpu().numpy()
    assert np.all(cov[:, :, :2, 2:] == 0) and np.all(cov[:, :, 2:, :2] == 0)
    assert np.array_equal(cov, np.swapaxes(cov, -1, -2))
    fb.close()
    fn = DeviceFit(Y, Xm, Xc, c, 1.0, orc.NAIVE)
    fn.sweep()
    torch.cuda.synchronize()
    cov = fn.Xc.cpu().numpy()
    offd = cov - np.einsum("ntd,de->ntde", np.diagonal(cov, axis1=-2, axis2=-1), np.eye(c["d"]))
    assert np.all(offd == 0) and np.all(np.diagonal(cov, axis1=-2, axis2=-1) > 0)
    fn.close()


def test_error_behaviour():
    from gpu_util import make_config
    from tame_b200 import _lib
    import ctypes as C
    lib = _lib.load()
    c = orc.model_constants(10, 3, 2)
    cfg, keep = make_config(c, 1.0, orc.GOOD)
    cfg.r = 9
    h = C.c_void_p()
    assert lib.tame_create(C.byref(cfg), C.byref(h)) == -1 and b"latent_dim" in lib.tame_last_error()
    cfg.r = 2
    _lib.check(lib.tame_create(C.byref(cfg), C.byref(h)))
    assert lib.tame_sweep(h) == -3          # nothing bound yet
    lib.tame_destroy(h)
    from src.models import TemporalAMEModel
    from src.inference import TemporalAMEStructuredMFVI
    m = TemporalAMEModel(n_nodes=8, n_time=3)
    m.generate_data()
    with pytest.raises(ValueError):
        TemporalAMEStructuredMFVI(m, factorization="invalid")


def test_device_generator_distribution_and_mirror():
    """tame_generate_Y: zero diagonal, mirror consistency (test_models.py:138-142), residual covariance ~ R,
    and shard-independence (rows generated separately equal the rows of the full array)."""
    from src.models import TemporalAMEModel
    m = TemporalAMEModel(n_nodes=96, n_time=12, latent_dim=3, rho_dyadic=0.6)
    Y = m.generate_data_device(seed=5).cpu().numpy()
    n = m.n
    assert np.all(Y[np.arange(n), np.arange(n)] == 0)
    assert np.array_equal(Y[:, :, :, 1], np.swapaxes(Y[:, :, :, 0], 0, 1))
    X = m.X.numpy()
    res = []
    for t in range(m.T):
        mu = orc.compute_mean(X[:, t, :2], X[:, t, 2:], m.r)
        iu = np.triu_indices(n, 1)
        res.append((Y[:, :, t] - mu)[iu])
    res = np.concatenate(res)
    cov = np.cov(res.T)
    assert np.allclose(cov, m.R.numpy(), atol=0.004), cov
    part = m.generate_data_device(seed=5, row_begin=32, row_end=64).cpu().numpy()
    assert np.array_equal(part, Y[32:64])


@pytest.mark.parametrize("path", ["device-loop", "device-loop-nh1", "host-loop"])
def test_fit_batch_matches_per_fit_oracle(path, monkeypatch):
    """BASELINE config 5 in miniature: a grid of independent small fits (n, T, r, ar, rho vary; all three methods) through
    tame_fit_batch, each compared with the oracle's fit() including the per-fit early stop.  Default path: one launch of the
    whole-fit kernel per fit (k_fit, both team shapes); TAME_BATCH=host: the host-driven loop."""
    from gpu_util import run_batch
    monkeypatch.delenv("TAME_BATCH", raising=False)
    monkeypatch.delenv("TAME_NH", raising=False)
    if path == "host-loop":
        monkeypatch.setenv("TAME_BATCH", "host")
    elif path == "device-loop-nh1":
        monkeypatch.setenv("TAME_NH", "1")
    grid = [(10, 5, 0.8, 0.5, 2), (24, 8, 0.5, 0.0, 2), (40, 3, 0.9, 0.8, 2), (33, 12, 0.3, -0.3, 2), (70, 4, 0.8, 0.5, 2),
            (12, 20, 0.7, 0.2, 2), (130, 7, 0.8, 0.5, 8), (96, 33, 0.6, 0.3, 3)]
    fits = []
    for k, (n, T, ar, rho, r) in enumerate(grid):
        for meth in (("naive", "good") if r == 2 else ("good", "bad")):
            c, Y, Xm, Xc = random_problem(n, T, r, seed=300 + k, rho=rho, ar=ar)
            fits.append((c, Y, Xm, Xc, 0.05 if meth == "bad" else 0.3, orc.MODE_OF[meth]))
    max_iter, tol = 12, 2e-2
    traces, n_done, states, launches = run_batch(fits, max_iter, tol, n_streams=4)
    if path == "host-loop":
        assert launches > 2 * len(fits)
    else:
        assert launches == 2 * len(fits), "one k_hab and one k_fit per fit"
    stopped_early = 0
    for f, (c, Y, Xm, Xc, lr, mode) in enumerate(fits):
        Om, Oc = Xm.copy(), Xc.copy()
        oel, oms = orc.fit(Y, Om, Oc, c, lr, mode, max_iter, tol, blocked=(c["n"] > 80))
        assert n_done[f] == len(oel), (f, n_done[f], len(oel))
        stopped_early += len(oel) < max_iter
        assert trace_ok(traces[f][0], oel) and trace_ok(traces[f][1], oms)
        assert rel_err(states[f][0], Om) < TOL and rel_err(states[f][1], Oc) < TOL
    assert stopped_early > 0, "the test should exercise the per-fit early stop"


@pytest.mark.parametrize("variant", ["mma", "dfma"])
@pytest.mark.parametrize("shape", [(96, 33, 4), (129, 6, 8), (200, 40, 8)])
def test_elbo_pass_variants_agree_with_oracle(shape, variant, monkeypatch):
    """Both implementations of the fused ELBO/MSE pass -- FP64 tensor-core (DMMA) tiles and the DFMA ring -- on mirror-
    consistent Y (triangular pass) and on a perturbed Y (full pass)."""
    from gpu_util import DeviceFit
    monkeypatch.setenv("TAME_LLMSE", variant)
    n, T, r = shape
    c, Y, Xm, Xc = random_problem(n, T, r, seed=4242 + n)
    for asym in (False, True):
        Yt = Y.copy()
        if asym:
            Yt[5, 60, 1, 1] -= 0.25
        f = DeviceFit(Yt, Xm, Xc, c, 0.3, orc.GOOD)
        got = f.elbo_mse()
        f.close()
        ref = list(orc.elbo_parts(Yt, Xm, Xc, c, orc.GOOD))
        assert abs(got[1] - ref[0]) <= TOL * abs(ref[0]), (variant, asym, got[1], ref[0])
        mse = orc.reconstruction_mse(Yt, Xm, c)
        assert abs(got[5] - mse) <= TOL * abs(mse)


@pytest.mark.parametrize("meth", ["good", "naive"])
def test_hundred_sweeps_no_drift(meth, sweep_path):
    """The chain carries its inverse by rank-2 Woodbury updates between refreshes (every TAME_REFRESH nodes); 100 sweeps on
    a shape with several refresh windows and streaming sub-blocks must still sit on the oracle's literal Gauss-Seidel
    schedule: whole ELBO / MSE traces and the final state at rel 1e-9."""
    from gpu_util import fit_host
    n, T, r, iters = 200, 12, 4, 100
    c, Y, Xm, Xc = random_problem(n, T, r, seed=77, rho=0.5)
    lr, mode = 0.3, orc.MODE_OF[meth]
    el, ms, Gm, Gc = fit_host(Y, Xm, Xc, c, lr, mode, iters)
    Om, Oc = Xm.copy(), Xc.copy()
    oel, oms = [], []
    for _ in range(iters):
        orc.sweep_fast(Y, Om, Oc, c, lr, mode)
        oel.append(orc.elbo(Y, Om, Oc, c, mode))
        oms.append(orc.reconstruction_mse(Y, Om, c))
    assert rel_err(Gm, Om) < TOL, rel_err(Gm, Om)
    assert rel_err(Gc, Oc) < TOL, rel_err(Gc, Oc)
    assert trace_ok(el, oel) and trace_ok(ms, oms)


def test_deterministic_mode_is_bitwise_reproducible(monkeypatch):
    """TAME_DETERMINISTIC=1 fixes the summation order of the streamed partner sums (no convoy start position): two runs of the
    same fit give bit-identical traces and state (the default order depends on timing at the 1e-16 level)."""
    from gpu_util import fit_host
    monkeypatch.setenv("TAME_DETERMINISTIC", "1")
    c, Y, Xm, Xc = random_problem(700, 5, 2, seed=5, rho=0.4)
    a = fit_host(Y, Xm, Xc, c, 0.3, orc.GOOD, 3)
    b = fit_host(Y, Xm, Xc, c, 0.3, orc.GOOD, 3)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
