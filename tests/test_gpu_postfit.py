"""The post-fit step (csrc/tame_align.cu) against plain high-precision references: Procrustes / sign alignment and the
contribution / U'V-correlation diagnostics, at every latent width, across the index boundaries of the kernels and on
degenerate inputs.

Alignment.  The reference is oracle/align_oracle.py: float64 NumPy with LAPACK's SVD, the routine the golden fixtures
pin.  A rotation R = U V' of svd(M) is only defined where M is: element by element comparisons are made where the
oracle's singular values have sigma_min > 1e-6 sigma_max and, when det(U V') < 0, a gap above 1e-3 sigma_max between the two
smallest (the reference negates the smallest singular direction).  Elsewhere (rank-deficient estimates, n < k) R is
not unique and LAPACK's choice is not the device's, so properties are checked: R orthogonal with det +1, the objective
tr(M'R) equal to the oracle's (the optimum value is unique even where R is not), and the output equal to what the
device's own R gives.  Tolerances: rel 1e-9 on outputs and errors, 1e-12 on orthogonality and det.

Diagnostics.  The reference is the literal n x n evaluation of the reference module (every a_i + b_j and U_i.V_j), in
extended precision (`lit_step`): np.longdouble where it is wider than double, else math.fsum over the float64 terms.
The kernels use Gram identities instead (sum_ij (U_i.V_j)^2 = <U'U, V'V>, ...), which cancel when the states carry a
large common offset.  In float64 that cancellation stays below 6e-13 rel for the additive contribution at an offset of
100x the spread of a and b (about 1.5e-10 at 1000x; it reaches 1e-9 near 3000x), and below 2e-13 abs for the
correlation with U and V offset by 10x their spread.  The gauge tests stay within those offsets.  Tolerances: rel 1e-9
on contributions and the state error, abs 1e-9 on correlations.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import align_oracle as ao
from oracle import diag_oracle as do

TOL = 1e-9
ORTH = 1e-12
EXT = np.finfo(np.longdouble).eps < np.finfo(np.float64).eps
MSE_CAP = 2048 * 1184          # tame_state_mse: 2048 elements a block up to 8 blocks per SM on 148 SMs, then grid-stride


def _cuda(x, dev="cuda"):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def _np(x):
    return x.detach().cpu().numpy()


def _close(a, b, tol=TOL):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and float(np.max(np.abs(a - b), initial=0.0)) <= tol * max(1e-300, float(np.max(np.abs(b), initial=0.0)))


@pytest.fixture
def f64():
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    yield
    torch.set_default_dtype(old)


# ---- alignment helpers ------------------------------------------------------------------------------------------------

def _orth(rng, k, m=None, proper=False):
    """Random orthogonal k x k matrices (m of them, or one); proper=True: det +1."""
    Q, Rq = np.linalg.qr(rng.standard_normal((m or 1, k, k)))
    Q = Q * np.sign(np.diagonal(Rq, axis1=-2, axis2=-1))[:, None, :]
    if proper:
        Q[np.linalg.det(Q) < 0, :, 0] *= -1
    return Q if m else Q[0]


def _classify(Ms):
    """(well_posed, reflected) flags of (m, k, k) matrices from the oracle's SVD.  Well posed: the oracle's rotation is
    unique and stable, so the output is compared element by element."""
    U, s, Vt = np.linalg.svd(Ms)
    refl = np.linalg.det(U @ Vt) < 0
    ok = s[:, -1] > 1e-6 * s[:, 0]
    if Ms.shape[-1] > 1:
        ok &= ~refl | (s[:, -2] - s[:, -1] > 1e-3 * s[:, 0])
    return ok, refl


def _well_posed(M):
    return bool(_classify(M[None])[0][0])


def _reflected(M):
    return bool(_classify(M[None])[1][0])


def _check_rotation(R, M):
    """Properties every rotation has: orthogonal, det +1, the optimal objective tr(M'R)."""
    _check_orthogonal(R[None])
    Ro = ao.procrustes_rotation(M, np.eye(M.shape[0]))         # svd of I' M
    scale = float(np.linalg.svd(M, compute_uv=False).sum())
    assert abs(float(np.trace(M.T @ R)) - float(np.trace(M.T @ Ro))) <= 1e-12 * scale


def _check_orthogonal(Rs):
    k = Rs.shape[-1]
    assert float(np.abs(Rs @ Rs.transpose(0, 2, 1) - np.eye(k)).max()) < ORTH
    assert float(np.abs(np.linalg.det(Rs) - 1.0).max()) < ORTH


def _cross(Xe, Xt, r, each):
    """The matrices the device takes rotations of, in the order of its rotation output: (T * 2, r, r) = X_true' X_est of
    the U and V block of every time step, or (1, 2r, 2r) of the temporal means."""
    if not each:
        return (Xt.mean(axis=1)[:, 2:].T @ Xe.mean(axis=1)[:, 2:])[None]
    U, V = slice(2, 2 + r), slice(2 + r, 2 + 2 * r)
    Ms = np.stack([np.einsum("ntk,ntc->tkc", Xt[:, :, c], Xe[:, :, c]) for c in (U, V)], axis=1)
    return Ms.reshape(-1, r, r)


def _device_align(Xe, Xt, r, each, dev="cuda"):
    """(aligned, mse, rotations) from the library, through _align_states_device and through the C ABI with the rotation
    buffer; the two must agree bit for bit."""
    from tame_b200 import _lib
    from tame_b200 import alignment as al
    e, t = _cuda(Xe, dev), _cuda(Xt, dev)
    out, mse = al._align_states_device(e, t, r, each, True)
    n, T, _ = Xe.shape
    k, nrot = (r, 2 * T) if each else (2 * r, 1)
    rot = torch.empty(nrot, k, k, dtype=torch.float64, device=dev)
    out2 = torch.empty_like(e)
    m2 = C.c_double(0.0)
    with torch.cuda.device(e.device):
        _lib.check(_lib.load().tame_align_states(n, T, r, e.data_ptr(), t.data_ptr(), int(each), out2.data_ptr(),
                                                 rot.data_ptr(), C.byref(m2), torch.cuda.current_stream(e.device).cuda_stream))
    assert torch.equal(out2, out) and m2.value == mse
    return _np(out), mse, _np(rot)


def check_alignment(Xe, Xt, r, each):
    """Device alignment of (n, T, 2+2r) states against the oracle.  Returns (well-posed flag, det < 0 flag) per matrix."""
    out, mse, rot = _device_align(Xe, Xt, r, each)
    Ms = _cross(Xe, Xt, r, each)
    ok, refl = _classify(Ms)
    _check_orthogonal(rot)
    for m in np.flatnonzero(~ok):
        _check_rotation(rot[m], Ms[m])
    expected = np.empty_like(Xe)                  # what the device's own rotations give
    expected[..., :2] = ao.align_signs_rows(Xe[..., :2], Xt[..., :2])
    if each:
        good_t = ok.reshape(-1, 2).all(axis=1)
        for b in range(2):
            cols = slice(2 + b * r, 2 + (b + 1) * r)
            expected[:, :, cols] = ao.align_signs_rows(np.einsum("ntk,tkc->ntc", Xe[:, :, cols], rot[b::2]), Xt[:, :, cols])
    else:
        good_t = np.full(Xe.shape[1], ok[0])
        expected[..., 2:] = ao.align_signs_rows(Xe[..., 2:] @ rot[0], Xt[..., 2:])
    assert np.isfinite(out).all()
    assert _close(out, expected)
    ref = ao.align_temporal_states(Xe, Xt, r, align_each_time=each)
    assert _close(out[:, good_t], ref[:, good_t])
    ref_mse = float((((ref if good_t.all() else out) - Xt) ** 2).mean())
    assert abs(mse - ref_mse) <= TOL * ref_mse
    return ok, refl


def check_procrustes(Xe, Xt, well_posed=None):
    """tame_procrustes without and with scaling against the oracle; returns whether M was well posed."""
    from src.utils import procrustes_alignment
    M = Xt.T @ Xe
    ok = _well_posed(M) if well_posed is None else well_posed
    for scaling in (False, True):
        out, R = procrustes_alignment(_cuda(Xe), _cuda(Xt), scaling=scaling)
        out, R = _np(out), _np(R)
        assert np.isfinite(out).all()
        _check_rotation(R, M)
        ref, Ro = ao.procrustes_alignment(Xe, Xt, scaling=scaling)
        if ok:
            assert _close(R, Ro) and _close(out, ref)
        else:                                     # what the device's own R gives
            mine = Xe @ R
            if scaling:
                num, den = float(np.trace(Xt.T @ mine)), float(np.trace(mine.T @ mine))
                mine = mine * (num / den) if den > 1e-10 else mine
            assert _close(out, mine)
    return ok


def rotated_states(n, T, r, each, seed):
    """Truth with separated column scales; estimate = truth rotated (per time step and block, or one 2r x 2r rotation
    for the global mode), rows sign-flipped at random, plus noise.  Rotations have either determinant."""
    rng = np.random.default_rng(seed)
    d = 2 + 2 * r
    Xt = rng.standard_normal((n, T, d))
    Xt[..., 2:] *= np.sqrt(1.0 + np.tile(np.arange(r), 2))
    Xe = Xt.copy()
    Xe[..., :2] *= rng.choice([-1.0, 1.0], (n, T, 1))
    if each:
        for b in range(2):
            cols = slice(2 + b * r, 2 + (b + 1) * r)
            Xe[:, :, cols] = np.einsum("ntk,tkc->ntc", Xt[:, :, cols], _orth(rng, r, T)) * rng.choice([-1.0, 1.0], (n, T, 1))
    else:
        Xe[..., 2:] = (Xt[..., 2:] @ _orth(rng, 2 * r)) * rng.choice([-1.0, 1.0], (n, T, 1))
    return Xe + 0.3 * rng.standard_normal(Xe.shape), Xt


# (n, T, r, align_each_time): every r in both modes; n = 1, 2, 3, 5 (warps without rows, the 4-node DMMA group, n < k),
# 63/64/65 (the 64-row split), 257, 777, 2049; T on both sides of the 32-step slice of k_align_apply; T = 4800 makes
# split_rows collapse to one split and leaves k_align_apply 8 blocks per 32-step column
ALIGN_CASES = [(1, 33, 1, True), (2049, 2, 1, False), (63, 100, 2, True), (5, 31, 2, False), (65, 32, 3, True),
               (257, 65, 3, False), (777, 1, 4, True), (64, 33, 4, False), (2, 65, 5, True), (2049, 31, 5, False),
               (257, 33, 6, True), (3, 100, 6, False), (5, 2, 7, True), (777, 32, 7, False), (257, 4800, 8, True),
               (64, 65, 8, False), (2049, 100, 8, True)]
# (n, k) for tame_procrustes: every width, ragged second DMMA tile (k = 9..15) above n = 30, n < k at k = 3, 13, 16
PROC_CASES = [(1, 1), (2049, 2), (2, 3), (63, 4), (64, 5), (65, 6), (257, 7), (777, 8), (2049, 9), (63, 10), (64, 11),
              (65, 12), (3, 13), (257, 14), (777, 15), (5, 16)]


def procrustes_inputs(n, k, seed):
    rng = np.random.default_rng(seed)
    Xt = rng.standard_normal((n, k)) * np.sqrt(1.0 + np.arange(k))
    return Xt @ _orth(rng, k) + 0.3 * rng.standard_normal((n, k)), Xt


def _case_seed(*a):
    return int(sum((i + 1) * 7919 * int(v) for i, v in enumerate(a))) % 2**31


def test_alignment_matrix_is_mostly_compared_element_by_element():
    """The well-posedness rule must leave most matrices of the width x mode matrix to the element by element path (CPU)."""
    good = total = 0
    for n, T, r, each in ALIGN_CASES:
        Xe, Xt = rotated_states(n, T, r, each, _case_seed(n, T, r, each))
        ok = _classify(_cross(Xe, Xt, r, each))[0]
        good += int(ok.sum())
        total += ok.size
    for n, k in PROC_CASES:
        Xe, Xt = procrustes_inputs(n, k, _case_seed(n, k))
        good += _well_posed(Xt.T @ Xe)
        total += 1
    assert good >= 0.75 * total, (good, total)


@pytest.mark.gpu
@pytest.mark.parametrize("n,T,r,each", ALIGN_CASES)
def test_align_states_width_mode_matrix(n, T, r, each):
    Xe, Xt = rotated_states(n, T, r, each, _case_seed(n, T, r, each))
    ok, _ = check_alignment(Xe, Xt, r, each)
    if n >= 2 * r:
        assert ok.mean() >= 0.99
    if each:
        from src.utils import compute_alignment_error
        out, mse, _ = _device_align(Xe, Xt, r, each)
        err, al = compute_alignment_error(_cuda(Xe), _cuda(Xt), latent_dim=r)
        assert err == mse and np.array_equal(_np(al), out)


@pytest.mark.gpu
@pytest.mark.parametrize("n,k", PROC_CASES)
def test_procrustes_every_width(n, k):
    Xe, Xt = procrustes_inputs(n, k, _case_seed(n, k))
    ok = check_procrustes(Xe, Xt)
    assert ok or n < k


# ---- the reflection branch at size ------------------------------------------------------------------------------------

def _reflected_block(rng, n, k):
    """(truth, Q): an (n, k) truth with column scales sqrt(1..k) and Q = a rotation times diag(1, .., 1, -1).  The
    cross-covariance of the truth with truth @ Q (+ small noise) has singular values of about n * (1..k) and a polar
    factor with det -1."""
    D = np.ones(k)
    D[-1] = -1.0
    return rng.standard_normal((n, k)) * np.sqrt(np.arange(1, k + 1)), _orth(rng, k, proper=True) * D


@pytest.mark.gpu
@pytest.mark.parametrize("r", range(1, 9))
@pytest.mark.parametrize("each", [True, False])
def test_reflection_branch_at_size(r, each):
    """Both blocks of every time step (or the one 2r x 2r rotation) need the det < 0 correction, n >= 1000."""
    rng = np.random.default_rng(100 + r + 10 * each)
    n, T, d = 1000 + 131 * r, 3, 2 + 2 * r
    Xt = np.empty((n, T, d))
    Xe = np.empty((n, T, d))
    Xt[..., :2] = rng.standard_normal((n, T, 2))
    Xe[..., :2] = Xt[..., :2] * rng.choice([-1.0, 1.0], (n, T, 1)) + 0.3 * rng.standard_normal((n, T, 2))
    if each:
        for t in range(T):
            for b in range(2):
                cols = slice(2 + b * r, 2 + (b + 1) * r)
                Xt[:, t, cols], Q = _reflected_block(rng, n, r)
                Xe[:, t, cols] = Xt[:, t, cols] @ Q + 0.01 * rng.standard_normal((n, r))
    else:                           # the global mode rotates by the polar factor of the temporal means
        base, Q = _reflected_block(rng, n, 2 * r)
        for t in range(T):
            Xt[:, t, 2:] = base + 0.1 * rng.standard_normal((n, 2 * r))
            Xe[:, t, 2:] = Xt[:, t, 2:] @ Q + 0.01 * rng.standard_normal((n, 2 * r))
    ok, refl = check_alignment(Xe, Xt, r, each)
    assert ok.all() and refl.all()


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(1, 17))
def test_procrustes_reflection_branch_at_size(k):
    rng = np.random.default_rng(200 + k)
    Xt, Q = _reflected_block(rng, 1000 + 61 * k, k)
    Xe = Xt @ Q + 0.01 * rng.standard_normal(Xt.shape)
    M = Xt.T @ Xe
    assert _reflected(M) and _well_posed(M)
    assert check_procrustes(Xe, Xt)


# ---- rank-deficient estimates and n < k -------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("k", range(2, 17))
def test_procrustes_rank_deficient(k):
    rng = np.random.default_rng(300 + k)
    for rank in sorted({1, (k + 1) // 2, k - 1}):
        n = 200 + 37 * rank
        Xt = rng.standard_normal((n, k))
        Xe = rng.standard_normal((n, rank)) @ rng.standard_normal((rank, k))
        assert not _well_posed(Xt.T @ Xe)
        check_procrustes(Xe, Xt, well_posed=False)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 3])
@pytest.mark.parametrize("k", [8, 16])
def test_procrustes_fewer_nodes_than_width(n, k):
    rng = np.random.default_rng(400 + n + k)
    Xe, Xt = rng.standard_normal((n, k)), rng.standard_normal((n, k))
    assert not _well_posed(Xt.T @ Xe)
    check_procrustes(Xe, Xt, well_posed=False)


@pytest.mark.gpu
@pytest.mark.parametrize("n,each", [(2, True), (3, True), (2, False), (3, False), (300, True), (300, False)])
def test_align_states_rank_deficient(n, each):
    """r = 8: k = 8 per block or 16 for the global mode.  n = 2, 3 have fewer nodes than k; at n = 300 the estimate's
    multiplicative blocks have rank 1..k-1."""
    rng = np.random.default_rng(500 + n + each)
    r, T = 8, 5
    Xt = rng.standard_normal((n, T, 2 + 2 * r))
    Xe = rng.standard_normal((n, T, 2 + 2 * r))
    if n > 2 * r:
        B = rng.standard_normal((5, 2 * r))      # global mode: one row space for every step, so the mean has rank 5
        for t in range(T):
            if each:
                for b in range(2):
                    rank = 1 + (3 * t + b) % (r - 1)
                    Xe[:, t, 2 + b * r:2 + (b + 1) * r] = rng.standard_normal((n, rank)) @ rng.standard_normal((rank, r))
            else:
                Xe[:, t, 2:] = rng.standard_normal((n, 5)) @ B
    ok, _ = check_alignment(Xe, Xt, r, each)
    assert not ok.any()


# ---- ill-conditioned and clustered singular values -------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("k", range(2, 17))
@pytest.mark.parametrize("kind", ["cond1e10", "cluster1e-6"])
def test_procrustes_ill_conditioned_and_clustered(k, kind):
    """M = U diag(s) V' with det(U V') = +1.  cond1e10: s = 1 .. 0.1 and one s = 1e-10 (the polar factor's condition is
    2 / (s_{k-1} + s_k), so it stays well-conditioned); cluster1e-6: all s within 1e-6 relative.  R and the output
    are compared with the oracle even though the singular vectors themselves are ill-determined."""
    rng = np.random.default_rng(600 + k + 50 * (kind == "cond1e10"))
    if kind == "cond1e10":
        s = np.append(np.linspace(1.0, 0.1, k - 1), 1e-10)
    else:
        s = 1.0 + 1e-6 * rng.random(k)
    U, V = _orth(rng, k, proper=True), _orth(rng, k, proper=True)
    M = (U * s) @ V.T
    Qn = np.linalg.qr(rng.standard_normal((64 + k, k)))[0]
    Xt, Xe = Qn, Qn @ M
    check_procrustes(Xe, Xt, well_posed=True)


# ---- diagnostics: the extended-precision literal reference ------------------------------------------------------------

def _ld(x):
    return np.asarray(x, dtype=np.longdouble if EXT else np.float64)


def _sum(x):
    return x.sum() if EXT else math.fsum(np.ravel(x))


def lit_step(Xe, Xt, r, chunk=512):
    """Literal n x n sums of one time step, (n, 2+2r) states, in extended precision: every a_i + b_j and U_i.V_j is
    formed.  Returns dict(add_excl, add_incl, mul_excl, mul_incl) of Xe and, with Xt, corr = the Pearson correlation of
    the flattened products U V' of Xt and Xe (NaN where either variance is 0, like np.corrcoef)."""
    n = Xe.shape[0]
    a, b, Ue, Ve = _ld(Xe[:, 0]), _ld(Xe[:, 1]), _ld(Xe[:, 2:2 + r]), _ld(Xe[:, 2 + r:])
    s = dict(add_all=0, add_off=0, mul_all=0, mul_off=0, de=0, dt=0, dee=0, dtt=0, det=0)
    N = n * n
    if Xt is not None:          # the single pass runs over products shifted by their float64 mean: no cancellation
        Ut, Vt = _ld(Xt[:, 2:2 + r]), _ld(Xt[:, 2 + r:])
        she = float(Xe[:, 2:2 + r].sum(0) @ Xe[:, 2 + r:].sum(0)) / N
        sht = float(Xt[:, 2:2 + r].sum(0) @ Xt[:, 2 + r:].sum(0)) / N
    for i0 in range(0, n, chunk):
        i1 = min(n, i0 + chunk)
        diag = (np.arange(i1 - i0), np.arange(i0, i1))
        add = (a[i0:i1, None] + b[None, :]) ** 2
        pe = Ue[i0:i1] @ Ve.T
        mul = pe ** 2
        s["add_all"] += _sum(add)
        s["mul_all"] += _sum(mul)
        add[diag] = 0
        mul[diag] = 0
        s["add_off"] += _sum(add)
        s["mul_off"] += _sum(mul)
        if Xt is not None:
            de, dt = pe - she, Ut[i0:i1] @ Vt.T - sht
            s["de"] += _sum(de)
            s["dt"] += _sum(dt)
            s["dee"] += _sum(de * de)
            s["dtt"] += _sum(dt * dt)
            s["det"] += _sum(de * dt)
    out = dict(add_incl=float(s["add_all"] / N), mul_incl=float(s["mul_all"] / N),
               add_excl=float(s["add_off"] / (N - n)) if n > 1 else math.nan,
               mul_excl=float(s["mul_off"] / (N - n)) if n > 1 else math.nan)
    if Xt is not None:
        cov = s["det"] - s["de"] * s["dt"] / N
        ve, vt = s["dee"] - s["de"] ** 2 / N, s["dtt"] - s["dt"] ** 2 / N
        out["corr"] = float(min(1, max(-1, cov / np.sqrt(ve * vt)))) if ve > 0 and vt > 0 else math.nan
    return out


def lit_steps(Xe, Xt, r, ts):
    return [lit_step(Xe[:, t], None if Xt is None else Xt[:, t], r) for t in ts]


def _lit_job(args):
    return lit_step(*args)


def lit_steps_parallel(Xe, Xt, r, ts):
    """lit_steps over spawned worker processes, one per time step (the literal sums of an n = 8192 step take seconds)."""
    from gpu_util import oracle_pool
    with oracle_pool(len(ts)) as pool:
        return list(pool.map(_lit_job, [(np.ascontiguousarray(Xe[:, t]), np.ascontiguousarray(Xt[:, t]), r) for t in ts]))


def diag_states(n, T, r, seed):
    rng = np.random.default_rng(seed)
    Xt = rng.standard_normal((n, T, 2 + 2 * r))
    Xe = 0.8 * Xt + 0.4 * rng.standard_normal(Xt.shape) + 0.05
    return Xe, Xt


def device_diag(Xe, Xt, r):
    """{add_excl, add_incl, mul_excl, mul_incl, corr}: (T,) float64 arrays from the library."""
    from tame_b200 import diagnostics as dg
    e, t = _cuda(Xe), _cuda(Xt)
    out = {}
    for tag, excl in (("excl", True), ("incl", False)):
        add, mul = dg._contrib_device(e, r, excl)
        out["add_" + tag], out["mul_" + tag] = _np(add), _np(mul)
    out["corr"] = dg.compute_uv_correlation_over_time(e, t, r).double().numpy()
    return out


def check_diag(dev, refs, ts):
    for j, t in enumerate(ts):
        for q in ("add_excl", "add_incl", "mul_excl", "mul_incl"):
            assert abs(dev[q][t] - refs[j][q]) <= TOL * abs(refs[j][q]), (q, t, dev[q][t], refs[j][q])
        assert abs(dev["corr"][t] - refs[j]["corr"]) <= TOL, (t, dev["corr"][t], refs[j]["corr"])


@pytest.mark.parametrize("n,r", [(2, 1), (3, 4), (7, 2), (12, 8), (40, 5)])
def test_literal_reference_matches_diag_oracle(n, r):
    """The extended-precision reference is pinned to the float64 literal oracle (CPU)."""
    Xe, Xt = diag_states(n, 3, r, n + r)
    ref = lit_steps(Xe, Xt, r, range(3))
    add_x, mul_x = do.temporal_contributions(Xe, r, True)
    add_i, mul_i = do.temporal_contributions(Xe, r, False)
    corr = do.uv_correlation_over_time(Xe, Xt, r)
    for t in range(3):
        for q, v in (("add_excl", add_x), ("add_incl", add_i), ("mul_excl", mul_x), ("mul_incl", mul_i)):
            assert abs(ref[t][q] - v[t]) <= 1e-13 * abs(v[t])
        assert abs(ref[t]["corr"] - corr[t]) <= 1e-13
    Xt[:, 1, 2:2 + r] = 0.0                 # no U'V product: both say NaN
    with np.errstate(invalid="ignore", divide="ignore"):
        assert math.isnan(lit_step(Xe[:, 1], Xt[:, 1], r)["corr"]) and math.isnan(do.uv_correlation_over_time(Xe, Xt, r)[1])


# (n, T, r): every r; n = 2, 3, 5 (fewer rows than warps), 64/65, 777, 2049; T = 1, 31, 33 (one, a full and a ragged
# 32-step slice).  Both exclude_diagonal settings run on every case.
DIAG_CASES = [(2, 31, 1), (3, 33, 2), (5, 1, 3), (64, 33, 4), (65, 31, 5), (777, 1, 6), (2049, 33, 7), (2049, 31, 8),
              (5, 33, 8), (65, 1, 1), (777, 33, 2), (3, 31, 6), (64, 1, 7), (2, 33, 3), (777, 31, 4), (5, 31, 5)]


def _diag_ts(n, T):
    return list(range(T)) if n * n * T <= 300000 else sorted({t for t in (0, 1, T // 2, 31, T - 1) if t < T})


@pytest.mark.gpu
@pytest.mark.parametrize("n,T,r", DIAG_CASES)
def test_diagnostics_matrix(n, T, r, f64):
    Xe, Xt = diag_states(n, T, r, _case_seed(n, T, r))
    ts = _diag_ts(n, T)
    check_diag(device_diag(Xe, Xt, r), lit_steps(Xe, Xt, r, ts), ts)


@pytest.mark.gpu
def test_diagnostics_config4_size(f64):
    """n = 8192, T = 128, r = 8 (BASELINE config 4), checked at 4 time steps spread over both halves of the slices."""
    n, T, r = 8192, 128, 8
    Xe, Xt = diag_states(n, T, r, 4)
    ts = [0, 31, 64, 127]
    dev = device_diag(Xe, Xt, r)
    check_diag(dev, lit_steps_parallel(Xe, Xt, r, ts), ts)


@pytest.mark.gpu
@pytest.mark.parametrize("n,T,r", [(777, 33, 3), (65, 31, 8), (2049, 2, 1)])
def test_diagnostics_gauge_offsets(n, T, r, f64):
    """a -> a + c, b -> b - c leaves every a_i + b_j unchanged: the additive contributions keep their value for
    c = 0, 1, 10, 100 times the spread.  U and V with a common offset of up to 10x their spread: contributions and
    correlations against the literal sums of the offset states."""
    Xe0, Xt0 = diag_states(n, T, r, _case_seed(n, T, r, 1))
    ts = _diag_ts(n, T)
    base = lit_steps(Xe0, None, r, ts)
    spread = float(Xe0[..., :2].std())
    for c in (0, 1, 10, 100):
        Xe = Xe0.copy()
        Xe[..., 0] += c * spread
        Xe[..., 1] -= c * spread
        refs = lit_steps(Xe, None, r, ts)
        from tame_b200 import diagnostics as dg
        for excl, tag in ((True, "add_excl"), (False, "add_incl")):
            add = _np(dg._contrib_device(_cuda(Xe), r, excl)[0])
            for j, t in enumerate(ts):
                assert abs(add[t] - refs[j][tag]) <= TOL * refs[j][tag], (c, tag, t)
                assert abs(add[t] - base[j][tag]) <= TOL * base[j][tag], (c, tag, t)
    spread = float(Xe0[..., 2:].std())
    for m in (1, 3, 10):
        Xe, Xt = Xe0.copy(), Xt0.copy()
        Xe[..., 2:] += m * spread
        Xt[..., 2:] += m * spread
        check_diag(device_diag(Xe, Xt, r), lit_steps(Xe, Xt, r, ts), ts)


@pytest.mark.gpu
@pytest.mark.parametrize("count", [1, MSE_CAP - 1, MSE_CAP, MSE_CAP + 1, 8192 * 128 * 18])
def test_state_prediction_error_counts(count):
    """Grid sizes up to the 1184-block cap and the grid-stride loop past it; config 4 has 18.9 M elements."""
    from src.utils import compute_state_prediction_error
    g = torch.Generator(device="cuda").manual_seed(count)
    A = torch.randn(count, generator=g, dtype=torch.float64, device="cuda")
    B = 0.9 * A + torch.randn(count, generator=g, dtype=torch.float64, device="cuda") + 0.1
    ref = float(_sum((_ld(_np(A)) - _ld(_np(B))) ** 2) / count)
    assert abs(compute_state_prediction_error(A, B) - ref) <= TOL * ref


@pytest.mark.gpu
def test_state_prediction_error_broadcast_config4():
    from src.utils import compute_state_prediction_error
    n, T, d = 8192, 128, 18
    g = torch.Generator(device="cuda").manual_seed(8)
    A = torch.randn(n, T, d, generator=g, dtype=torch.float64, device="cuda")
    B = torch.randn(n, 1, d, generator=g, dtype=torch.float64, device="cuda")
    ref = float(_sum((_ld(_np(A)) - _ld(_np(B))) ** 2) / A.numel())
    assert abs(compute_state_prediction_error(A, B) - ref) <= TOL * ref
    assert abs(compute_state_prediction_error(B, A) - ref) <= TOL * ref


# ---- degenerate diagnostics -------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("n,T,r", [(65, 33, 3), (777, 40, 8), (5, 12, 1)])
def test_uv_correlation_of_zero_products_is_nan(n, T, r, f64):
    """A zero U or V block (of the truth, of the estimate, or one of each) leaves that time step's U V' products all
    zero: the correlation there is undefined (NaN, as torch.corrcoef and the reference return), and the other time
    steps do not change."""
    Xe0, Xt0 = diag_states(n, T, r, _case_seed(n, T, r, 2))
    U, V = slice(2, 2 + r), slice(2 + r, 2 + 2 * r)
    Xe, Xt = Xe0.copy(), Xt0.copy()
    zero = {0: [(Xt, U)], 5: [(Xt, V)], 7: [(Xe, U)], T - 1: [(Xe, V)], 3: [(Xt, U), (Xe, V)], 9: [(Xt, U), (Xt, V), (Xe, U)]}
    for t, parts in zero.items():
        for X, cols in parts:
            X[:, t, cols] = 0.0
    from tame_b200 import diagnostics as dg
    before = dg.compute_uv_correlation_over_time(_cuda(Xe0), _cuda(Xt0), r).double().numpy()
    corr = dg.compute_uv_correlation_over_time(_cuda(Xe), _cuda(Xt), r).double().numpy()
    others = [t for t in range(T) if t not in zero]
    assert np.isnan(corr[sorted(zero)]).all(), corr[sorted(zero)]
    assert np.array_equal(corr[others], before[others])
    ts = sorted(zero) + others[:3]
    refs = lit_steps(Xe, Xt, r, ts)
    for j, t in enumerate(ts):
        assert (math.isnan(refs[j]["corr"]) and math.isnan(corr[t])) or abs(corr[t] - refs[j]["corr"]) <= TOL
    # a truth without a multiplicative part, through both entry points
    from src.utils import compute_uv_product_correlation
    Xt = Xt0.copy()
    Xt[..., 2:] = 0.0
    assert np.isnan(dg.compute_uv_correlation_over_time(_cuda(Xe0), _cuda(Xt), r).numpy()).all()
    assert math.isnan(compute_uv_product_correlation(_cuda(Xe0[:, 0, 2:]), torch.zeros(n, 2 * r, device="cuda"), r))
    # the zero blocks still have well-defined contributions: the multiplicative one is 0 exactly
    add, mul = dg._contrib_device(_cuda(Xe), r, True)
    assert float(_np(mul)[7]) == 0.0 and float(_np(mul)[T - 1]) == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("T,r", [(1, 1), (33, 4), (5, 8)])
def test_contributions_of_one_node(T, r, f64):
    """n = 1 without the diagonal has no pair: NaN, as the literal reference's 0 / 0.  With the diagonal it is the one
    term."""
    from tame_b200 import diagnostics as dg
    X = np.random.default_rng(T + r).standard_normal((1, T, 2 + 2 * r))
    add, mul = dg._contrib_device(_cuda(X), r, True)
    assert torch.isnan(add).all() and torch.isnan(mul).all()
    add, mul = dg._contrib_device(_cuda(X), r, False)
    refs = lit_steps(X, None, r, range(T))
    assert _close(_np(add), [q["add_incl"] for q in refs]) and _close(_np(mul), [q["mul_incl"] for q in refs])
    from src.utils import compute_additive_contribution, compute_multiplicative_contribution
    assert math.isnan(compute_additive_contribution(torch.from_numpy(X[:, 0, :2])))
    assert math.isnan(compute_multiplicative_contribution(torch.from_numpy(X[:, 0, 2:])))


# ---- plumbing ---------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_cpu_float32_inputs_keep_dtype_and_device():
    """The reference's default dtype is float32: CPU float32 inputs come back as CPU float32 (the device computes in
    float64, so the result is the float64 answer for the float32 inputs, rounded once)."""
    from src.utils import (align_temporal_states, compute_alignment_error, compute_temporal_contributions,
                           compute_uv_correlation_over_time, procrustes_alignment)
    assert torch.get_default_dtype() == torch.float32
    Xe, Xt = rotated_states(70, 9, 3, True, 11)
    e32, t32 = torch.from_numpy(Xe).float(), torch.from_numpy(Xt).float()
    e64, t64 = e32.double().numpy(), t32.double().numpy()
    one_ulp = 2.0 ** -23
    out = align_temporal_states(e32, t32, 3)
    assert out.dtype == torch.float32 and out.device.type == "cpu"
    assert np.allclose(out.numpy(), ao.align_temporal_states(e64, t64, 3), rtol=one_ulp, atol=1e-30)
    err, al = compute_alignment_error(e32, t32, latent_dim=3)
    assert al.dtype == torch.float32 and not al.is_cuda and np.array_equal(al.numpy(), out.numpy())
    pa, R = procrustes_alignment(e32[:, 0, 2:5], t32[:, 0, 2:5])
    assert pa.dtype == R.dtype == torch.float32 and not pa.is_cuda and not R.is_cuda
    assert np.allclose(R.numpy(), ao.procrustes_rotation(e64[:, 0, 2:5], t64[:, 0, 2:5]), rtol=one_ulp, atol=1e-7)
    add, mul = compute_temporal_contributions(e32, 3)
    corr = compute_uv_correlation_over_time(e32, t32, 3)
    assert add.dtype == mul.dtype == corr.dtype == torch.float32 and not corr.is_cuda
    refs = lit_steps(e64, t64, 3, range(9))
    assert np.allclose(add.numpy(), [q["add_excl"] for q in refs], rtol=one_ulp, atol=0)
    assert np.allclose(corr.numpy(), [q["corr"] for q in refs], rtol=0, atol=one_ulp)


@pytest.mark.gpu
def test_non_contiguous_views(f64):
    from src.utils import (align_temporal_states, compute_state_prediction_error, compute_temporal_contributions,
                           compute_uv_correlation_over_time, procrustes_alignment)
    Xe, Xt = rotated_states(90, 12, 2, True, 12)
    # (T, n, d) storage seen as (n, T, d), every second time step of a (n, 2T, d) array
    e = _cuda(np.ascontiguousarray(Xe.transpose(1, 0, 2))).transpose(0, 1)
    t = torch.zeros(90, 24, 6, dtype=torch.float64, device="cuda")[:, ::2]
    t.copy_(_cuda(Xt))
    assert not e.is_contiguous() and not t.is_contiguous()
    assert _close(_np(align_temporal_states(e, t, 2)), ao.align_temporal_states(Xe, Xt, 2))
    assert _close(_np(align_temporal_states(e, t, 2, align_each_time=False)), ao.align_temporal_states(Xe, Xt, 2, False))
    refs = lit_steps(Xe, Xt, 2, range(12))
    add, mul = compute_temporal_contributions(e, 2)
    assert _close(add.numpy(), [q["add_excl"] for q in refs]) and _close(mul.numpy(), [q["mul_excl"] for q in refs])
    assert np.allclose(compute_uv_correlation_over_time(e, t, 2).numpy(), [q["corr"] for q in refs], rtol=0, atol=TOL)
    m = float(((Xe - Xt) ** 2).mean())
    assert abs(compute_state_prediction_error(t, e) - m) <= TOL * m
    pe, pt = e[:, 3, 2:], t[:, 3, 2:]                      # strided (n, 4) matrices
    out, R = procrustes_alignment(pe, pt)
    ref, Ro = ao.procrustes_alignment(Xe[:, 3, 2:], Xt[:, 3, 2:])
    assert _close(_np(R), Ro) and _close(_np(out), ref)


@pytest.mark.gpu
def test_side_stream_right_after_the_inputs_are_produced(f64):
    """Inputs written by kernels queued on a side stream, the call made on that stream before anything synchronises:
    the library must run on the caller's current stream."""
    from src.utils import align_temporal_states, compute_temporal_contributions, compute_uv_correlation_over_time
    n, T, r = 2049, 65, 4
    Xe, Xt = rotated_states(n, T, r, True, 13)
    src_e, src_t = _cuda(Xe), _cuda(Xt)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        big = torch.randn(4096, 4096, dtype=torch.float64, device="cuda")
        for _ in range(4):                      # keep the side stream busy before the inputs are written
            big = torch.tanh(big @ big)
        e, t = torch.empty_like(src_e), torch.empty_like(src_t)
        e.copy_(src_e)
        t.copy_(src_t)
        out = align_temporal_states(e, t, r)
        add, mul = compute_temporal_contributions(e, r)
        corr = compute_uv_correlation_over_time(e, t, r)
        out_h = _np(out)
    torch.cuda.synchronize()
    assert _close(out_h, ao.align_temporal_states(Xe, Xt, r))
    dev = device_diag(Xe, Xt, r)
    assert np.array_equal(add.numpy(), dev["add_excl"]) and np.array_equal(corr.numpy(), dev["corr"])


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [0, 1, -2, -1])
def test_align_signs_3d(dim):
    from src.utils import align_signs
    rng = np.random.default_rng(14 + dim)
    Xt = rng.standard_normal((7, 5, 6))
    shape = [1, 1, 1]
    shape[dim] = Xt.shape[dim]
    Xe = Xt * rng.choice([-1.0, 1.0], shape) + 0.5 * rng.standard_normal(Xt.shape)
    out = align_signs(torch.from_numpy(Xe), torch.from_numpy(Xt), dim=dim)
    assert np.array_equal(out.numpy(), ao.align_signs(Xe, Xt, dim=dim))
    out = align_signs(_cuda(Xe), _cuda(Xt), dim=dim)
    assert out.is_cuda and np.array_equal(_np(out), ao.align_signs(Xe, Xt, dim=dim))


@pytest.mark.gpu
def test_second_gpu_gives_the_same_result(f64):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from tame_b200 import diagnostics as dg
    n, T, r = 777, 33, 5
    Xe, Xt = rotated_states(n, T, r, True, 15)
    for each in (True, False):
        o0, m0, r0 = _device_align(Xe, Xt, r, each, "cuda:0")
        o1, m1, r1 = _device_align(Xe, Xt, r, each, "cuda:1")
        assert np.array_equal(o0, o1) and m0 == m1 and np.array_equal(r0, r1)
    for excl in (True, False):
        a0, b0 = dg._contrib_device(_cuda(Xe, "cuda:0"), r, excl)
        a1, b1 = dg._contrib_device(_cuda(Xe, "cuda:1"), r, excl)
        assert a1.device.index == 1 and np.array_equal(_np(a0), _np(a1)) and np.array_equal(_np(b0), _np(b1))
    c0 = dg.compute_uv_correlation_over_time(_cuda(Xe, "cuda:0"), _cuda(Xt, "cuda:0"), r)
    c1 = dg.compute_uv_correlation_over_time(_cuda(Xe, "cuda:1"), _cuda(Xt, "cuda:1"), r)
    assert torch.equal(c0, c1)
