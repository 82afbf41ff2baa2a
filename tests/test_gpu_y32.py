"""float32 observations kept as float32 on the device (tame_bind_Y_f32, tame_fit_batch_f32, tame_fit_host_f32,
tame_generate_Y_f32, and the drop-in classes on float32 models).

Every kernel that reads Y widens each dyad to FP64 right after the load and then runs the FP64 arithmetic unchanged,
so on the same float32 data the float32-storage path must equal the FP64 path run on Y.double(): bit for bit under
TAME_DETERMINISTIC=1 (the sweep's partner sums in a fixed order), within rel 1e-12 without it.  Both sides run here,
with the same team shape, sweep path, ELBO-pass variant and column-part count."""
import ctypes as C
import pickle

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, METHODS, golden_constants, load_golden
from gpu_util import DeviceFit, DeviceFit32, fit_host, make_config, random_problem, run_batch
from oracle import tame_oracle as orc

pytestmark = pytest.mark.gpu
LR = {"naive": 0.3, "good": 0.3, "bad": 0.05}
SWITCHES = ("TAME_BATCH", "TAME_SWEEP", "TAME_NH", "TAME_DETERMINISTIC", "TAME_NPARTS", "TAME_BATCH_STREAMS", "TAME_LLMSE",
            "TAME_SYMMETRIC")


@pytest.fixture(autouse=True)
def _deterministic(monkeypatch):
    for v in SWITCHES:
        monkeypatch.delenv(v, raising=False)
    monkeypatch.setenv("TAME_DETERMINISTIC", "1")


def _lib():
    from tame_b200 import _lib
    return _lib


# ---- float32 counterparts of the gpu_util helpers (the float64 side uses gpu_util itself) -----------------------
def fit_host32(Y, Xm, Xc, c, lr, mode, max_iter, tol=0.0):
    """gpu_util.fit_host through tame_fit_host_f32 (Y as float32 host memory)"""
    L = _lib()
    lib = L.load()
    cfg, keep = make_config(c, lr, mode)
    Y = np.ascontiguousarray(Y, dtype=np.float32)
    Xm = np.ascontiguousarray(Xm, dtype=np.float64).copy()
    Xc = np.ascontiguousarray(Xc, dtype=np.float64).copy()
    el, ms, nd = np.zeros(max(max_iter, 1)), np.zeros(max(max_iter, 1)), C.c_int32(0)
    L.check(lib.tame_fit_host_f32(C.byref(cfg), Y.ctypes.data, Xm.ctypes.data, Xc.ctypes.data, max_iter, float(tol),
                                  L.dptr(el), L.dptr(ms), C.byref(nd)))
    return el[:nd.value], ms[:nd.value], Xm, Xc


def run_batch32(fits, max_iter, tol, n_streams=0):
    """gpu_util.run_batch through tame_fit_batch_f32 (every Y as a float32 CUDA tensor)"""
    L = _lib()
    lib = L.load()
    nf = len(fits)
    cfgs = (L.TameConfig * nf)()
    Yp, Mp, Cp = (C.c_void_p * nf)(), (C.c_void_p * nf)(), (C.c_void_p * nf)()
    keep, dev = [], []
    for f, (c, Y, Xm, Xc, lr, mode) in enumerate(fits):
        cfgs[f], kk = make_config(c, lr, mode)
        keep.append(kk)
        t = [torch.as_tensor(np.ascontiguousarray(Y, dtype=np.float32)).cuda()] + \
            [torch.as_tensor(np.array(a, dtype=np.float64)).cuda() for a in (Xm, Xc)]
        dev.append(t)
        Yp[f], Mp[f], Cp[f] = t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr()
    torch.cuda.synchronize()
    el, ms, nd = np.zeros((nf, max_iter)), np.zeros((nf, max_iter)), (C.c_int32 * nf)()
    before = lib.tame_launch_count()
    L.check(lib.tame_fit_batch_f32(nf, cfgs, Yp, Mp, Cp, max_iter, tol, L.dptr(el), L.dptr(ms), nd, n_streams))
    launches = lib.tame_launch_count() - before
    n_done = np.array(list(nd))
    traces = [(el[f, :n_done[f]], ms[f, :n_done[f]]) for f in range(nf)]
    states = [(t[1].cpu().numpy(), t[2].cpu().numpy()) for t in dev]
    return traces, n_done, states, launches


def _handle_fit(c, Y, Xm, Xc, lr, mode, iters, y32, tol=0.0):
    """tame_fit on one handle (Y bound as float32 or float64); returns traces, n_done, ELBO parts, state, symmetric flag."""
    lib = _lib().load()
    f = DeviceFit32(Y, Xm, Xc, c, lr, mode) if y32 else DeviceFit(Y, Xm, Xc, c, lr, mode)
    try:
        el, ms, nd = np.zeros(iters), np.zeros(iters), C.c_int32(0)
        _lib().check(lib.tame_fit(f.h, iters, tol, _lib().dptr(el), _lib().dptr(ms), C.byref(nd)))
        parts = f.elbo_mse()
        return dict(el=el[:nd.value], ms=ms[:nd.value], nd=nd.value, parts=parts, Xm=f.Xm.cpu().numpy(),
                    Xc=f.Xc.cpu().numpy(), sym=lib.tame_y_symmetric(f.h))
    finally:
        f.close()


def _same(a, b, exact=True):
    assert a["nd"] == b["nd"], (a["nd"], b["nd"])
    for k in ("el", "ms", "parts", "Xm", "Xc"):
        if exact:
            assert np.array_equal(a[k], b[k]), (k, np.max(np.abs(a[k] - b[k])))
        else:
            assert np.all(np.abs(a[k] - b[k]) <= 1e-12 * np.max(np.abs(b[k]))), (k, np.max(np.abs(a[k] - b[k])))


def _pair(c, Y32, Xm, Xc, lr, mode, iters, tol=0.0, exact=True):
    """the float32-storage fit against the FP64 fit of the widened Y; returns the float32 side"""
    Y32 = np.ascontiguousarray(Y32, dtype=np.float32)
    a = _handle_fit(c, Y32, Xm, Xc, lr, mode, iters, True, tol)
    b = _handle_fit(c, Y32.astype(np.float64), Xm, Xc, lr, mode, iters, False, tol)
    _same(a, b, exact)
    assert a["sym"] == b["sym"]
    return a


# ---- golden cases, both team shapes and the stream-ordered panel path ------------------------------------------
@pytest.mark.parametrize("variant", ["nh1", "nh2", "panel"])
@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_golden_f32_equals_f64(case, variant, monkeypatch):
    if variant == "panel":
        monkeypatch.setenv("TAME_SWEEP", "panel")
    else:
        monkeypatch.setenv("TAME_NH", variant[-1])
    g = load_golden(case)
    c = golden_constants(g)
    iters = min(int(g["max_iter"]), 12)
    for m in METHODS:
        a = _pair(c, g["Y"], g[f"{m}_init_mean"], g[f"{m}_init_cov"], float(g["lr"]), orc.MODE_OF[m], iters,
                  float(g["tolerance"]))
        assert a["sym"] == 1                       # the golden Y is mirror-consistent, and stays so rounded to float32


@pytest.mark.parametrize("llmse", ["mma", "dfma"])
@pytest.mark.parametrize("r", [4, 8])
def test_elbo_pass_variants(r, llmse, monkeypatch):
    monkeypatch.setenv("TAME_LLMSE", llmse)
    c, Y, Xm, Xc = random_problem(72, 40, r, seed=300 + r)
    for m in METHODS:
        _pair(c, Y, Xm, Xc, LR[m], orc.MODE_OF[m], 4)


# ---- latent dimensions x ragged shapes: n on both sides of 32 / 64, 1 / 2 / 4 column parts, T in {1, 7, 33} ----
SHAPES = {1: [(520, 1), (33, 7)], 2: [(65, 33), (200, 7)], 3: [(31, 7), (200, 1)], 4: [(520, 7), (64, 33)],
          5: [(63, 33), (20, 1)], 6: [(200, 33), (40, 7)], 7: [(33, 1), (520, 33)], 8: [(70, 7), (200, 33)]}


@pytest.mark.parametrize("r", sorted(SHAPES))
def test_shapes_f32_equals_f64(r):
    for k, (n, T) in enumerate(SHAPES[r]):
        m = METHODS[(r + k) % 3]
        c, Y, Xm, Xc = random_problem(n, T, r, seed=10 * r + k)
        _pair(c, Y, Xm, Xc, LR[m], orc.MODE_OF[m], 3)


def test_not_deterministic_rel_1e12(monkeypatch):
    """default summation order (convoy start of the streaming CTAs): the two storages agree to rel 1e-12"""
    monkeypatch.delenv("TAME_DETERMINISTIC")
    c, Y, Xm, Xc = random_problem(600, 33, 8, seed=77)
    _pair(c, Y, Xm, Xc, 0.3, orc.GOOD, 3, exact=False)


# ---- mirror check ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("comp", [0, 1])
def test_one_ulp_breaks_the_mirror(comp):
    """One float32 entry of a mirror-consistent Y moved by one ulp (either component of the lower-index side): the
    check reports 0, and the fit (full ELBO pass) still equals the FP64 fit of the same values."""
    c, Y, Xm, Xc = random_problem(70, 9, 3, seed=5)
    Y32 = Y.astype(np.float32)
    base = _pair(c, Y32, Xm, Xc, 0.3, orc.GOOD, 2)
    assert base["sym"] == 1
    i, j, t = 3, 41, 4
    Y32[i, j, t, comp] = np.nextafter(Y32[i, j, t, comp], np.float32(np.inf))
    a = _pair(c, Y32, Xm, Xc, 0.3, orc.GOOD, 2)
    assert a["sym"] == 0


def test_nonzero_diagonal():
    c, Y, Xm, Xc = random_problem(45, 7, 2, seed=6)
    Y32 = Y.astype(np.float32)
    Y32[np.arange(45), np.arange(45)] = np.float32(0.75)
    for m in METHODS:
        a = _pair(c, Y32, Xm, Xc, LR[m], orc.MODE_OF[m], 3)
        assert a["sym"] == 1                        # the diagonal is not part of the mirror property


def test_rebind_other_type():
    """one handle: bind float32, rebind float64, rebind float32; each state equals a fresh handle of that type"""
    lib = _lib().load()
    c, Y, Xm, Xc = random_problem(100, 12, 4, seed=8)
    Y32 = Y.astype(np.float32)
    Y64 = torch.as_tensor(Y32.astype(np.float64)).cuda()
    ref = _handle_fit(c, Y32, Xm, Xc, 0.3, orc.GOOD, 1, True)
    f = DeviceFit32(Y32, Xm, Xc, c, 0.3, orc.GOOD)
    try:
        _lib().check(lib.tame_bind_Y(f.h, Y64.data_ptr()))
        _lib().check(lib.tame_bind_Y_f32(f.h, f.Y.data_ptr()))
        f.sweep()
        out = f.elbo_mse()
        assert np.array_equal(f.Xm.cpu().numpy(), ref["Xm"]) and np.array_equal(out, ref["parts"])
    finally:
        f.close()


# ---- batches --------------------------------------------------------------------------------------------------
def test_batch_f32_equals_f64():
    fits = []
    for k, (n, T, r) in enumerate([(40, 16, 1), (200, 7, 3), (520, 2, 8), (33, 33, 4), (64, 1, 6)]):
        c, Y, Xm, Xc = random_problem(n, T, r, seed=900 + k)
        m = METHODS[k % 3]
        fits.append((c, Y.astype(np.float32), Xm, Xc, LR[m], orc.MODE_OF[m]))
    tr32, nd32, st32, l32 = run_batch32(fits, 6, 1e-4)
    tr64, nd64, st64, l64 = run_batch([(c, Y.astype(np.float64), Xm, Xc, lr, md) for c, Y, Xm, Xc, lr, md in fits], 6, 1e-4)
    assert l32 == 2 * len(fits) and l64 == 2 * len(fits)          # one k_hab + one k_fit per fit: no host loop
    assert np.array_equal(nd32, nd64)
    for f in range(len(fits)):
        for a, b in zip(tr32[f] + st32[f], tr64[f] + st64[f]):
            assert np.array_equal(a, b), f


def test_batch_f32_pooled_handles():
    """one stream: a pooled handle re-pointed across n = 192 / 512 gives what each fit gives on its own"""
    fits = []
    for k, (n, T, r, m) in enumerate([(192, 8, 2, "good"), (512, 8, 2, "bad"), (192, 16, 2, "naive"), (512, 4, 2, "good")]):
        c, Y, Xm, Xc = random_problem(n, T, r, seed=950 + k)
        fits.append((c, Y.astype(np.float32), Xm, Xc, LR[m], orc.MODE_OF[m]))
    tr, nd, st, launches = run_batch32(fits, 4, 0.0, n_streams=1)
    assert launches == 2 * len(fits)
    for f, fit in enumerate(fits):
        tr1, nd1, st1, _ = run_batch32([fit], 4, 0.0, n_streams=1)
        assert nd1[0] == nd[f]
        for a, b in zip(tr1[0] + st1[0], tr[f] + st[f]):
            assert np.array_equal(a, b), f


def test_fit_host_f32():
    c, Y, Xm, Xc = random_problem(90, 10, 5, seed=12)
    Y32 = Y.astype(np.float32)
    a = fit_host32(Y32, Xm, Xc, c, 0.3, orc.GOOD, 3)
    b = fit_host(Y32.astype(np.float64), Xm, Xc, c, 0.3, orc.GOOD, 3)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


# ---- generator ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,T,rows", [(50, 1, None), (70, 33, None), (70, 33, (13, 47))])
def test_generate_f32_is_rounded_f64(n, T, rows):
    lib = _lib().load()
    r = 3
    c = orc.model_constants(n, T, r)
    X = torch.randn(n, T, c["d"], dtype=torch.float64, generator=torch.Generator().manual_seed(n + T)).cuda()
    lo, hi = rows if rows else (0, n)
    R = np.ascontiguousarray(c["R"].reshape(4))
    Y64 = torch.empty(hi - lo, n, T, 2, dtype=torch.float64, device="cuda")
    Y32 = torch.empty(hi - lo, n, T, 2, dtype=torch.float32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    _lib().check(lib.tame_generate_Y(n, T, r, _lib().dptr(R), X.data_ptr(), C.c_uint64(7), lo, hi, Y64.data_ptr(), st))
    _lib().check(lib.tame_generate_Y_f32(n, T, r, _lib().dptr(R), X.data_ptr(), C.c_uint64(7), lo, hi, Y32.data_ptr(), st))
    torch.cuda.synchronize()
    assert torch.equal(Y32.view(torch.int32), Y64.float().view(torch.int32))
    if rows is None:
        assert torch.equal(Y32[..., 0], Y32.transpose(0, 1)[..., 1])       # mirror-consistent bit for bit


def test_generate_data_device_dtype():
    from tame_b200 import TemporalAMEModel
    m = TemporalAMEModel(n_nodes=40, n_time=6, latent_dim=2, seed=3)
    Y = m.generate_data_device(dtype=torch.float32, seed=5)
    assert Y.dtype == torch.float32 and m.Y is Y
    Y64 = m.generate_data_device(seed=5)
    assert Y64.dtype == torch.float64 and torch.equal(Y, Y64.float())
    with pytest.raises(ValueError):
        m.generate_data_device(dtype=torch.float16)


# ---- drop-in classes ------------------------------------------------------------------------------------------
def _model(n=48, T=9, r=3):
    from tame_b200 import TemporalAMEModel
    torch.manual_seed(0)
    m = TemporalAMEModel(n_nodes=n, n_time=T, latent_dim=r, seed=1)
    m.generate_data()
    return m


def test_dropin_float32_storage_and_parity():
    from tame_b200 import TemporalAMEStructuredMFVI
    m32 = _model()
    assert m32.Y.dtype == torch.float32
    m32.Y = m32.Y.cuda()
    ptr = m32.Y.data_ptr()
    m64 = _model()
    m64.Y = m64.Y.double()
    a = TemporalAMEStructuredMFVI(m32, factorization="good", learning_rate=0.3)
    b = TemporalAMEStructuredMFVI(m64, factorization="good", learning_rate=0.3)
    ha, hb = a.fit(max_iter=4, verbose=False), b.fit(max_iter=4, verbose=False)
    assert a._engine.Y.dtype == torch.float32 and a._engine.Y.data_ptr() == ptr     # bound without a copy
    assert b._engine.Y.dtype == torch.float64
    assert ha == hb
    assert torch.equal(a.X_mean, b.X_mean) and torch.equal(a.X_cov, b.X_cov)
    assert a._compute_expected_log_likelihood() == b._compute_expected_log_likelihood()


def test_dropin_pickle_resume():
    from tame_b200 import TemporalAMENaiveMFVI
    straight = TemporalAMENaiveMFVI(_model(), learning_rate=0.3)
    straight.fit(max_iter=4, tolerance=0.0, verbose=False)
    vi = TemporalAMENaiveMFVI(_model(), learning_rate=0.3)
    vi.fit(max_iter=2, tolerance=0.0, verbose=False)
    vi2 = pickle.loads(pickle.dumps(vi))
    vi2.fit(max_iter=2, tolerance=0.0, verbose=False)
    assert vi2._engine.Y.dtype == torch.float32
    assert vi2.history == straight.history
    assert torch.equal(vi2.X_mean, straight.X_mean) and torch.equal(vi2.X_cov, straight.X_cov)


@pytest.mark.parametrize("mixed", [False, True])
def test_fit_batch_each_equals_its_own_fit(mixed):
    from tame_b200 import TemporalAMENaiveMFVI, TemporalAMEStructuredMFVI, fit_batch

    def make():
        out = []
        for k, (n, T, r) in enumerate([(30, 5, 2), (70, 12, 4), (40, 33, 1)]):
            m = _model(n, T, r)
            if mixed and k == 1:
                m.Y = m.Y.double()
            cls = TemporalAMENaiveMFVI if k == 2 else TemporalAMEStructuredMFVI
            out.append(cls(m, learning_rate=0.3))
        return out
    batch, own = make(), make()
    fit_batch(batch, max_iter=5, tolerance=1e-6)
    for vb, vo in zip(batch, own):
        # the whole-fit kernel sums the ELBO in its own order: the host loop's results within rel 1e-9, as for float64
        vo.fit(max_iter=5, tolerance=1e-6, verbose=False)
        vo._pull()
        for k in ("elbo", "reconstruction_error"):
            a, b = np.array(vb.history[k]), np.array(vo.history[k])
            assert a.shape == b.shape and np.all(np.abs(a - b) <= 1e-9 * np.abs(b)), k
        for x, y in zip(vb._exact, vo._exact):
            assert torch.allclose(x, y, rtol=1e-9, atol=1e-12)


def test_multi_gpu_float32_equals_single():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from tame_b200 import TemporalAMEStructuredMFVI
    one = TemporalAMEStructuredMFVI(_model(128, 8, 2), factorization="good", learning_rate=0.3, device="cuda:0")
    two = TemporalAMEStructuredMFVI(_model(128, 8, 2), factorization="good", learning_rate=0.3, devices=[0, 1])
    h1, h2 = one.fit(max_iter=3, verbose=False), two.fit(max_iter=3, verbose=False)
    assert all(Yr.dtype == torch.float32 for Yr in two._engine.Y)
    e1, e2 = np.array(h1["elbo"]), np.array(h2["elbo"])
    assert np.all(np.abs(e1 - e2) <= 1e-9 * np.abs(e1)), (e1, e2)
    one._pull(), two._pull()
    assert torch.allclose(one._exact[0], two._exact[0], rtol=1e-9, atol=1e-12)


# ---- errors ---------------------------------------------------------------------------------------------------
def test_bind_f32_null_arguments():
    lib = _lib().load()
    assert lib.tame_bind_Y_f32(None, 1) == -1
    assert b"null" in lib.tame_last_error()
    c, Y, Xm, Xc = random_problem(20, 3, 1, seed=1)
    f = DeviceFit32(Y, Xm, Xc, c, 0.3, orc.GOOD)
    try:
        assert lib.tame_bind_Y_f32(f.h, None) == -1
        assert b"null" in lib.tame_last_error()
        assert lib.tame_bind_Y(f.h, None) == -1
    finally:
        f.close()
