"""The ELBO/MSE pass of tame_elbo_mse (k_llmse / k_llmse_mma -> k_cellterms -> k_reduce6 -> k_finalize), the mirror
check k_symcheck that picks its SYM path, and the whole-fit kernel's own pass (tame_llmse_small), checked bit for bit.

Integer-valued inputs make the pass exact.  a, b, U, V are integers in [-2, 2] and Y = mu + e with integer residuals
|e| <= 3, so every product, FMA chain, DMMA, per-row moment sum, shuffle, grid.z partial and k_reduce6 sum is exact
whatever its order (all partial sums stay below 2^53: about 1e11 at config 4, where |Y| <= 39 is exact in float32 too).
R^-1 = [[1, 1/4], [1/4, 1/2]] is dyadic, so p0 S00 + 2q S01 + p1 S11 is exact, and logdet_R = -2 * LOG2PI (the
kernels' own double) makes k_finalize add exactly 0 for the constant.  The device must then return, bit for bit,
LL = -quad / 2 (naive mode) and MSE = sq / (n (n-1) T), where quad and sq are integer sums taken here from Y and the
latents alone: one dyad more or fewer, a wrong partner, a swapped U_i.V_j / U_j.V_i, a counted diagonal, tail partner
or lane, a z-range dropped or counted twice -- each changes an integer.  Good and bad modes add the trace term
0.1 tr(R^-1)/d (n-1) sum tr X_cov; with integer diagonals that sum is exact too and LL is held to 2 ulp of the formula.

The cell terms (LP0, LPT, H) on real-valued state are compared per term with a float64 NumPy evaluation per cell,
summed with math.fsum."""
import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

from conftest import METHODS
from oracle import tame_oracle as orc

gpu = pytest.mark.gpu
LOG2PI = 1.8378770664093454835606594728112      # the kernels' literal (one ulp above math.log(2 * math.pi))
RINV = np.array([[1.0, 0.25], [0.25, 0.5]])
SWITCHES = ("TAME_BATCH", "TAME_SWEEP", "TAME_NH", "TAME_DETERMINISTIC", "TAME_NPARTS", "TAME_BATCH_STREAMS", "TAME_LLMSE",
            "TAME_SYMMETRIC")


@pytest.fixture(autouse=True)
def _clean_env(monkeypatch):
    for v in SWITCHES:
        monkeypatch.delenv(v, raising=False)


# ---- integer problems ---------------------------------------------------------------------------------------------
def _hash(i, j, t, salt):
    """integer in [-3, 3] from the ORDERED pair (i, j) and t (int64 tensors that broadcast)"""
    h = (i * 0x2545F491 + j * 0x6C8E9CF5 + t * 0x1B873593 + salt) & 0xFFFFFFFF
    h = h ^ (h >> 15)
    h = (h * 0x2C1B3C6D) & 0xFFFFFFFF
    h = h ^ (h >> 12)
    return h % 7 - 3


def _means(Xm, lo, hi, r):
    """mu[i, j, t, 0] = a_i + b_j + U_i.V_j, mu[i, j, t, 1] = a_j + b_i + U_j.V_i for the rows lo..hi-1 (static_ame.py)"""
    a, b = Xm[:, :, 0], Xm[:, :, 1]
    U, V = Xm[:, :, 2:2 + r], Xm[:, :, 2 + r:]
    m0 = a[lo:hi, None, :] + b[None, :, :] + torch.einsum("itk,jtk->ijt", U[lo:hi], V)
    m1 = a[None, :, :] + b[lo:hi, None, :] + torch.einsum("jtk,itk->ijt", U, V[lo:hi])
    return m0, m1


def int_constants(n, T, r):
    c = orc.model_constants(n, T, r)
    c["R_inv"] = RINV.copy()
    c["logdet_R"] = -2.0 * LOG2PI
    return c


def int_state(n, T, r, seed, structure, device):
    """integer means in [-2, 2]; covariances (d+1) I + S with S symmetric in {-1, 0, 1} (SPD by Gershgorin), with the
    structure of the mode: full ('good'), zero cross blocks ('bad'), diagonal ('naive')"""
    d = 2 + 2 * r
    g = torch.Generator(device=device).manual_seed(seed)
    Xm = torch.randint(-2, 3, (n, T, d), generator=g, device=device).to(torch.float64)
    S = torch.randint(-1, 2, (n, T, d, d), generator=g, device=device, dtype=torch.int8).to(torch.float64)
    S = torch.triu(S) + torch.triu(S, 1).transpose(-1, -2)
    Xc = S + (d + 1) * torch.eye(d, dtype=torch.float64, device=device)
    del S
    if structure == "bad":
        Xc[..., :2, 2:] = 0.0
        Xc[..., 2:, :2] = 0.0
    elif structure == "naive":
        Xc = torch.diag_embed(torch.diagonal(Xc, dim1=-2, dim2=-1))
    return Xm.contiguous(), Xc.contiguous()


def int_Y(Xm, r, seed, mirror=True, dtype=torch.float64, chunk=64):
    """Y[i,j,t,0] = mu_ij + e(i,j,t), Y[i,j,t,1] = mu_ji + e(j,i,t): mirror-consistent by construction.  mirror=False
    draws channel 1 from a second hash, so Y[j,i,t,0] != Y[i,j,t,1] for most dyads.  The diagonal holds large
    integers that differ between the channels (the pass and the mirror check must ignore it)."""
    n, T = Xm.shape[0], Xm.shape[1]
    dev = Xm.device
    Y = torch.empty(n, n, T, 2, dtype=dtype, device=dev)
    j = torch.arange(n, device=dev)[None, :, None]
    t = torch.arange(T, device=dev)[None, None, :]
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        i = torch.arange(lo, hi, device=dev)[:, None, None]
        m0, m1 = _means(Xm, lo, hi, r)
        e0 = _hash(i, j, t, seed)
        e1 = _hash(j, i, t, seed) if mirror else _hash(j, i, t, seed + 7919)
        y0, y1 = m0 + e0, m1 + e1
        diag = (i == j)
        y0 = torch.where(diag, 1000.0 + (i % 5).to(torch.float64), y0)
        y1 = torch.where(diag, 1037.0 + (i % 5).to(torch.float64), y1)
        Y[lo:hi, :, :, 0] = y0.to(dtype)
        Y[lo:hi, :, :, 1] = y1.to(dtype)
    return Y


def exact_sums(Y, Xm, Xc, r, chunk=64):
    """Integer sums of the pass, from Y and the latents alone (structured_mf.py:124-146, temporal_ame.py:255-291):
    S00, S01, S11 = sum_{i<j,t} e0^2, e0 e1, e1^2; sq = sum_{i!=j,t} e0^2 + e1^2; tr = sum_{i,t} tr X_cov[i,t].
    The residuals are recomputed in FP64 (exact for these values) and asserted to be integers."""
    n = Y.shape[0]
    dev = Y.device
    cols = torch.arange(n, device=dev)
    s00 = s01 = s11 = sq = 0
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        rows = torch.arange(lo, hi, device=dev)
        m0, m1 = _means(Xm, lo, hi, r)
        e0 = Y[lo:hi, :, :, 0].to(torch.float64) - m0
        e1 = Y[lo:hi, :, :, 1].to(torch.float64) - m1
        del m0, m1
        assert torch.equal(e0, torch.round(e0)) and torch.equal(e1, torch.round(e1)), "residuals must be integers"
        e0, e1 = e0.to(torch.int64), e1.to(torch.int64)
        upper = (cols[None, :] > rows[:, None])[:, :, None]
        offd = (cols[None, :] != rows[:, None])[:, :, None]
        s00 += int(torch.sum(torch.where(upper, e0 * e0, 0)))
        s01 += int(torch.sum(torch.where(upper, e0 * e1, 0)))
        s11 += int(torch.sum(torch.where(upper, e1 * e1, 0)))
        sq += int(torch.sum(torch.where(offd, e0 * e0 + e1 * e1, 0)))
        del e0, e1
    trd = torch.diagonal(Xc, dim1=-2, dim2=-1)
    assert torch.equal(trd, torch.round(trd))
    tr = int(torch.sum(trd.to(torch.int64)))
    return dict(s00=s00, s01=s01, s11=s11, sq=sq, tr=tr)


def exact_quad(s):
    """p0 S00 + 2 q S01 + p1 S11 as an exact double (R^-1 is dyadic)"""
    p0, q, p1 = (Fraction(float(x)) for x in (RINV[0, 0], RINV[0, 1], RINV[1, 1]))
    qd = p0 * s["s00"] + 2 * q * s["s01"] + p1 * s["s11"]
    assert Fraction(float(qd)) == qd
    return float(qd)


def expected_ll_mse(s, n, T, d, mode):
    """(LL candidates, MSE): k_finalize's formula on the exact sums.  Naive mode has one exact value; the trace term may
    be contracted into an FMA, so good/bad give the plain and the fused evaluation."""
    quad = exact_quad(s)
    mse = float(s["sq"]) / (float(n) * float(n - 1) * float(T))
    if mode == orc.NAIVE:
        return [-0.5 * quad], mse
    k = 0.1 * (RINV[0, 0] + RINV[1, 1]) / float(d) * float(n - 1)
    plain = -0.5 * (quad + k * float(s["tr"]))
    fused = -0.5 * float(Fraction(quad) + Fraction(k) * s["tr"])
    return [plain, fused], mse


def check_out6(out, s, n, T, d, mode, what=""):
    lls, mse = expected_ll_mse(s, n, T, d, mode)
    assert out[5] == mse, (what, "MSE", out[5], mse)
    if mode == orc.NAIVE:
        assert out[1] == lls[0], (what, "LL", out[1], lls[0])
    else:
        assert min(abs(out[1] - v) for v in lls) <= 2 * math.ulp(lls[0]), (what, "LL", out[1], lls)
    assert out[0] == ((out[1] + out[2]) + out[3]) + out[4], (what, "ELBO", list(out))


# ---- launch geometry (restated from tame_ops.cu) --------------------------------------------------------------------
def llmse_z(n, T, sms):
    """grid.z of the DFMA pass (launch_llmse_tile): the partner range is split when the (time slice x 32-row tile) grid
    alone would leave SMs idle"""
    base = -(-T // 32) * -(-n // 32)
    return 1 if base >= 3 * sms else min(4, -(-3 * sms // base))


def llmse_zranges(n, jlo, z, JC=8):
    """the partner ranges [jbeg, jend) of the z-split (k_llmse): jlo is 0, or the tile's first chunk on the SYM path"""
    zlen = -(-(-(-(n - jlo) // z)) // JC) * JC
    return [(jlo + b * zlen, min(n, jlo + (b + 1) * zlen)) for b in range(z)]


def llmse_partials(n, T, sms, mma):
    return -(-T // 32) * -(-n // 16) if mma else -(-T // 32) * -(-n // 32) * llmse_z(n, T, sms)


def branch_shapes(sms):
    """(n, T) pairs that put the DFMA pass on grid.z = 1, 2, 3 and 4, each with a ragged twin (n and T off the tile)"""
    shapes = [(65, 33), (63, 31)]
    for z in (3, 2, 1):
        T = 256 if z == 1 else 128
        k = 1
        while llmse_z(32 * k, T, sms) != z:
            k += 1
        n = 32 * k
        shapes += [(n, T), (n - 4, T - 8)]
    return shapes


def slice_width(T):
    """W of tame_llmse_small: 8, 16 or 32 time steps per slice, whichever pads T least"""
    W = 32
    if -(-T // 16) * 16 < -(-T // W) * W:
        W = 16
    if -(-T // 8) * 8 < -(-T // W) * W:
        W = 8
    return W


# ---- device helpers -----------------------------------------------------------------------------------------------
def _lib():
    from tame_b200 import _lib as L
    return L


def _handle(c, Y, Xm, Xc, mode, lr=0.0):
    from gpu_util import DeviceFit, DeviceFit32
    return (DeviceFit32 if Y.dtype == torch.float32 else DeviceFit)(Y, Xm, Xc, c, lr, mode)


def _bind(f, Y):
    L = _lib()
    L.check(f.lib.tame_bind_Y_f32(f.h, Y.data_ptr()) if Y.dtype == torch.float32 else f.lib.tame_bind_Y(f.h, Y.data_ptr()))
    return f.lib.tame_y_symmetric(f.h)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def run_pass(c, Y, Xm, Xc, mode, s, monkeypatch, mirror, what):
    """tame_elbo_mse on Y (SYM path when mirror), checked exactly; a mirror Y again with TAME_SYMMETRIC=0, which must give
    the same bits.  Returns out6."""
    n, T, d = c["n"], c["T"], c["d"]
    f = _handle(c, Y, Xm, Xc, mode)
    try:
        sym = f.lib.tame_y_symmetric(f.h)
        assert sym == (1 if mirror else 0), (what, sym)
        out = f.elbo_mse()
        check_out6(out, s, n, T, d, mode, what)
        if mirror:
            monkeypatch.setenv("TAME_SYMMETRIC", "0")
            assert _bind(f, Y) == 0
            monkeypatch.delenv("TAME_SYMMETRIC")
            full = f.elbo_mse()
            assert np.array_equal(full, out), (what, "full pass differs from the SYM pass", full, out)
        return out
    finally:
        f.close()


# ---- 1. exact LL / MSE: every latent dimension, both ELBO-pass variants, both storages ----------------------------
VARIANTS = [("dfma", r) for r in range(1, 9)] + [("mma", 4), ("mma", 8)]
NS = [2, 3, 15, 16, 17, 31, 32, 33, 63, 64, 65, 129, 130]
TS = [1, 31, 32, 33, 65]


@gpu
@pytest.mark.parametrize("llmse,r", VARIANTS)
def test_exact_ll_mse(llmse, r, monkeypatch):
    """n crosses the 16-row DMMA tile, the 32-row DFMA tile and the 8-partner chunk; T crosses the 32-step slice.  Each
    shape: a mirror Y (SYM path, then the full pass), a non-mirror Y, in float32 and float64 storage; the two storages of
    the same values must give the same bits."""
    monkeypatch.setenv("TAME_LLMSE", llmse)
    k = VARIANTS.index((llmse, r))
    for s_ in range(6):
        n, T = NS[(6 * k + s_) % len(NS)], TS[(k + s_) % len(TS)]
        meth = METHODS[(k + s_) % 3]
        mode = orc.MODE_OF[meth]
        c = int_constants(n, T, r)
        Xm, Xc = int_state(n, T, r, seed=100 * k + s_, structure=meth, device="cuda")
        for mirror in (True, False):
            Y64 = int_Y(Xm, r, seed=17 * k + s_, mirror=mirror)
            s = exact_sums(Y64, Xm, Xc, r)
            outs = []
            for Y in (Y64, Y64.to(torch.float32)):
                outs.append(run_pass(c, Y, Xm, Xc, mode, s, monkeypatch, mirror,
                                     f"{llmse} r={r} n={n} T={T} {meth} mirror={mirror} {Y.dtype}"))
            assert np.array_equal(outs[0], outs[1]), (n, T, mirror, outs)


# ---- 2. launch branches: grid.z = 1..4, more than 256 partials, config 4 ------------------------------------------
def test_z_split_coverage_148_sms():
    """the branch shapes of the GPU test reach every grid.z of the DFMA pass on a 148-SM B200, and k_reduce6 walks more
    than its 256 threads' worth of partials on the large ones"""
    sms = 148
    shapes = branch_shapes(sms)
    zs = {sh: llmse_z(*sh, sms) for sh in shapes}
    assert zs[(1184, 128)] == 3 and zs[(1180, 120)] == 3
    assert zs[(1792, 128)] == 2 and zs[(1788, 120)] == 2
    assert zs[(1792, 256)] == 1 and zs[(1788, 248)] == 1
    assert zs[(65, 33)] == 4 and zs[(63, 31)] == 4
    assert set(zs.values()) == {1, 2, 3, 4}
    assert all(llmse_partials(n, T, sms, False) > 256 for n, T in shapes if n > 1000)
    assert llmse_partials(1184, 128, sms, True) > 256
    # every other shape in tests/ runs on z = 4, config 4 on z = 1
    assert llmse_z(2304, 33, sms) == 4 and llmse_z(8192, 128, sms) == 1
    # at z = 2 and 3 the rounding of the range length to whole 8-partner chunks leaves uneven and empty last ranges
    assert llmse_zranges(1184, 1152, 3) == [(1152, 1168), (1168, 1184), (1184, 1184)]
    assert llmse_zranges(1180, 1152, 3) == [(1152, 1168), (1168, 1180), (1184, 1180)]
    assert llmse_zranges(1788, 0, 2) == [(0, 896), (896, 1788)]
    for n, z in ((1184, 3), (1180, 3), (1792, 2), (1788, 2)):
        for jlo in range(0, n, 32):
            covered = [j for a, b in llmse_zranges(n, jlo, z) for j in range(a, b)]
            assert covered == list(range(jlo, n))


@gpu
def test_launch_branches(monkeypatch):
    sms = _sms()
    shapes = branch_shapes(sms)
    assert {llmse_z(n, T, sms) for n, T in shapes} == {1, 2, 3, 4}
    assert any(llmse_partials(n, T, sms, False) > 256 for n, T in shapes)
    for k, (n, T) in enumerate(shapes):
        r = 2 if k % 2 == 0 else 3
        c = int_constants(n, T, r)
        Xm, Xc = int_state(n, T, r, seed=500 + k, structure="naive", device="cuda")
        for mirror in (True, False):
            Y = int_Y(Xm, r, seed=900 + k, mirror=mirror, dtype=torch.float32 if (k + mirror) % 2 else torch.float64)
            s = exact_sums(Y, Xm, Xc, r)
            run_pass(c, Y, Xm, Xc, orc.NAIVE, s, monkeypatch, mirror, f"n={n} T={T} z={llmse_z(n, T, sms)}")
            del Y
        torch.cuda.empty_cache()


@gpu
@pytest.mark.parametrize("llmse,r", [("dfma", 8), ("mma", 4), ("mma", 8)])
def test_launch_branches_wide(llmse, r, monkeypatch):
    """the z = 3 shape at r = 8 (DFMA), and the DMMA tile at more than 256 partials; good mode (trace term)"""
    monkeypatch.setenv("TAME_LLMSE", llmse)
    sms = _sms()
    n, T = next(sh for sh in branch_shapes(sms) if llmse_z(*sh, sms) == 3)
    assert llmse_partials(n, T, sms, llmse == "mma") > 256
    c = int_constants(n, T, r)
    Xm, Xc = int_state(n, T, r, seed=r, structure="good", device="cuda")
    Y = int_Y(Xm, r, seed=31 + r, mirror=True, dtype=torch.float32)
    s = exact_sums(Y, Xm, Xc, r)
    run_pass(c, Y, Xm, Xc, orc.GOOD, s, monkeypatch, True, f"{llmse} r={r} n={n} T={T}")


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_config4_exact(dtype, monkeypatch):
    """config 4 itself (n = 8192, T = 128, r = 8; 69 GB of Y in float32, 137 GB in float64): one dyad is about 2e-10
    of the LL sum here, far below any relative tolerance, but not below an exact one.  Both ELBO-pass variants."""
    n, T, r = 8192, 128, 8
    d = 2 + 2 * r
    dev = torch.device("cuda", 0)
    need = n * n * T * 2 * torch.tensor([], dtype=dtype).element_size() + 3 * n * T * d * d * 8 + (8 << 30)
    torch.cuda.empty_cache()
    if torch.cuda.mem_get_info(dev)[0] < need:
        pytest.skip("not enough free HBM for config 4 in this storage")
    c = int_constants(n, T, r)
    Xm, Xc = int_state(n, T, r, seed=4, structure="good", device=dev)
    Y = int_Y(Xm, r, seed=44, mirror=True, dtype=dtype)
    s = exact_sums(Y, Xm, Xc, r, chunk=32)
    f = _handle(c, Y, Xm, Xc, orc.NAIVE)
    try:
        assert f.lib.tame_y_symmetric(f.h) == 1
        for llmse in ("dfma", "mma"):
            monkeypatch.setenv("TAME_LLMSE", llmse)
            check_out6(f.elbo_mse(), s, n, T, d, orc.NAIVE, f"config 4 {llmse} {dtype}")
    finally:
        f.close()
        del f, Y, Xm, Xc
        torch.cuda.empty_cache()


# ---- 3. mirror check ----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_mirror_check(dtype):
    """One asymmetric entry (moved by +1, so the SYM path would also get LL / MSE wrong) at the first dyad, an adjacent
    pair, the last dyad and the last (ragged) time step, from either side and in either channel: the flag is 0 and the
    full pass is exact.  +0.0 against -0.0 (equal values, different bits): flag 0.  Diagonal-only changes: flag 1."""
    n, T, r = 70, 33, 3
    d = 2 + 2 * r
    c = int_constants(n, T, r)
    Xm, Xc = int_state(n, T, r, seed=3, structure="naive", device="cuda")
    Y = int_Y(Xm, r, seed=5, mirror=True, dtype=dtype)
    s = exact_sums(Y, Xm, Xc, r)
    f = _handle(c, Y, Xm, Xc, orc.NAIVE)
    try:
        assert f.lib.tame_y_symmetric(f.h) == 1
        check_out6(f.elbo_mse(), s, n, T, d, orc.NAIVE, "mirror")
        spots = [(0, 1, 0), (1, 0, 0), (40, 41, 7), (41, 40, 7), (n - 2, n - 1, T - 1), (n - 1, n - 2, T - 1)]
        for (i, j, t) in spots:
            for ch in (0, 1):
                keep = Y[i, j, t, ch].clone()
                Y[i, j, t, ch] += 1
                assert _bind(f, Y) == 0, (i, j, t, ch)
                check_out6(f.elbo_mse(), exact_sums(Y, Xm, Xc, r), n, T, d, orc.NAIVE, f"({i},{j},{t},{ch})")
                Y[i, j, t, ch] = keep
        assert _bind(f, Y) == 1
        # +0.0 / -0.0: numerically a mirror image, not bit for bit
        for (i, j, t) in [(0, 1, 0), (40, 41, T - 1)]:
            keep = (Y[i, j, t, 0].clone(), Y[j, i, t, 1].clone())
            Y[i, j, t, 0] = 0.0
            Y[j, i, t, 1] = -0.0
            assert _bind(f, Y) == 0, (i, j, t)
            check_out6(f.elbo_mse(), exact_sums(Y, Xm, Xc, r), n, T, d, orc.NAIVE, f"-0.0 at ({i},{j},{t})")
            Y[i, j, t, 0], Y[j, i, t, 1] = keep
        # the diagonal is not part of the mirror property (int_Y already writes different channels there)
        idx = torch.arange(n, device=Y.device)
        Y[idx, idx, :, 0] = -7.0
        Y[idx, idx, :, 1] = 11.0
        Y[0, 0, T - 1, 1] = -0.0
        assert _bind(f, Y) == 1
        check_out6(f.elbo_mse(), s, n, T, d, orc.NAIVE, "diagonal")
    finally:
        f.close()


# ---- 4. cell terms on real-valued state ---------------------------------------------------------------------------
def cell_ref(Xm, Xc, c):
    """(LP0, LPT, H) and the sums of their terms' magnitudes, per cell in float64 (slogdet, einsum) and summed with
    math.fsum (structured_mf.py:148-209)"""
    T, d = Xm.shape[1], c["d"]
    L = orc.LOG_2PI
    ld = np.linalg.slogdet(Xc)[1]
    m0 = Xm[:, 0]
    q0 = np.einsum("ia,ab,ib->i", m0, c["S0_inv"], m0)
    t0 = np.einsum("ab,iba->i", c["S0_inv"], Xc[:, 0])
    lp0 = -0.5 * (c["logdet_S0"] + q0 + t0 + d * L)
    a0 = 0.5 * (abs(c["logdet_S0"]) + np.abs(q0) + np.abs(t0) + d * L)
    lpt, at = np.zeros(0), np.zeros(0)
    if T > 1:
        res = Xm[:, 1:] - Xm[:, :-1] @ c["Phi"].T
        qt = np.einsum("ita,ab,itb->it", res, c["Q_inv"], res)
        tt = np.einsum("ab,itba->it", c["Q_inv"], Xc[:, 1:])
        lpt = -0.5 * (c["logdet_Q"] + qt + tt + d * L)
        at = 0.5 * (abs(c["logdet_Q"]) + np.abs(qt) + np.abs(tt) + d * L)
    ent = 0.5 * (d * (1 + L) + ld)
    ae = 0.5 * (d * (1 + L) + np.abs(ld))
    f = lambda x: math.fsum(np.ravel(x).tolist())
    return [f(lp0), f(lpt), f(ent)], [f(a0), f(at), f(ae)]


def cell_wave_bound(r, sms):
    """an upper bound of the cells one resident wave of k_cellterms covers: SMs x 8 blocks (2048 threads) x 8 warps x G
    cells per warp (G = 4, 2, 1 for lane groups of 8, 16, 32)"""
    D = 2 + 2 * r
    return sms * 8 * 8 * (32 // (8 if D <= 8 else (16 if D <= 16 else 32)))


def cell_shapes(r, sms):
    """fewer cells than one block's pass, T = 1, and about three resident waves"""
    T = 200
    return [(17, 9), (33, 1), (-(-3 * cell_wave_bound(r, sms) // T), T)]


@gpu
@pytest.mark.parametrize("r", range(1, 9))
def test_cell_terms(r):
    sms = _sms()
    d = 2 + 2 * r
    for k, (n, T) in enumerate(cell_shapes(r, sms)):
        structure = METHODS[(r + k) % 3]
        rng = np.random.default_rng(10 * r + k)
        c = orc.model_constants(n, T, r)
        c["Phi"] = 0.8 * np.eye(d) + 0.05 * rng.standard_normal((d, d))        # not symmetric: the kernel's transposes
        Xm = 0.5 * rng.standard_normal((n, T, d))
        B = rng.standard_normal((n, T, d, d))
        Xc = B @ np.swapaxes(B, -1, -2) / d + 0.5 * np.eye(d)
        if structure == "bad":
            Xc[..., :2, 2:] = 0.0
            Xc[..., 2:, :2] = 0.0
        elif structure == "naive":
            Xc = Xc * np.eye(d)
        Y = torch.zeros(n, n, T, 2, dtype=torch.float64, device="cuda")
        f = _handle(c, Y, torch.as_tensor(Xm).cuda(), torch.as_tensor(Xc).cuda(), orc.MODE_OF[structure], lr=0.3)
        try:
            out = f.elbo_mse()
        finally:
            f.close()
        ref, mag = cell_ref(Xm, Xc, c)
        for name, got, want, m in zip(("LP0", "LPT", "H"), out[2:5], ref, mag):
            assert abs(got - want) <= 1e-12 * m, (r, n, T, structure, name, got, want, m)
        if T == 1:
            assert out[3] == 0.0
        assert out[0] == ((out[1] + out[2]) + out[3]) + out[4]
        del Y
    n, T = cell_shapes(r, sms)[-1]
    assert n * T >= 3 * cell_wave_bound(r, sms)


# ---- 5. the whole-fit kernel's own pass ----------------------------------------------------------------------------
FIT_CASES = [(2, 7, 1), (17, 48, 2), (65, 64, 4), (33, 33, 8), (130, 1, 3), (40, 16, 5), (31, 40, 6), (64, 32, 7)]


@gpu
def test_fit_kernel_pass(monkeypatch):
    """tame_fit_device with lr = 0 for one iteration leaves the state bit for bit; its MSE trace entry is then the exact
    value and its ELBO entry matches tame_elbo_mse on the same handle within rel 1e-13.  T selects every slice width."""
    assert {slice_width(T) for _, T, _ in FIT_CASES} == {8, 16, 32}
    for k, (n, T, r) in enumerate(FIT_CASES):
        meth = METHODS[k % 3]
        mode = orc.MODE_OF[meth]
        mirror = k % 2 == 0
        c = int_constants(n, T, r)
        Xm, Xc = int_state(n, T, r, seed=70 + k, structure=meth, device="cuda")
        Y = int_Y(Xm, r, seed=80 + k, mirror=mirror, dtype=torch.float32 if k % 4 < 2 else torch.float64)
        s = exact_sums(Y, Xm, Xc, r)
        lls, mse = expected_ll_mse(s, n, T, c["d"], mode)
        f = _handle(c, Y, Xm, Xc, mode, lr=0.0)
        try:
            assert f.lib.tame_y_symmetric(f.h) == (1 if mirror else 0)
            Xm0, Xc0 = Xm.clone(), Xc.clone()
            el = torch.zeros(1, dtype=torch.float64, device="cuda")
            ms = torch.zeros_like(el)
            nd = torch.zeros(1, dtype=torch.int32, device="cuda")
            _lib().check(f.lib.tame_fit_device(f.h, 1, 0.0, el.data_ptr(), ms.data_ptr(), nd.data_ptr()))
            torch.cuda.synchronize()
            assert int(nd.item()) == 1
            assert torch.equal(f.Xm, Xm0) and torch.equal(f.Xc, Xc0), "lr = 0 must leave the state unchanged"
            what = f"n={n} T={T} r={r} W={slice_width(T)} {meth}"
            assert float(ms.item()) == mse, (what, float(ms.item()), mse)
            out = f.elbo_mse()
            check_out6(out, s, n, T, c["d"], mode, what)
            assert abs(float(el.item()) - out[0]) <= 1e-13 * abs(out[0]), (what, float(el.item()), out[0])
        finally:
            f.close()


# ---- 6. the exact reference itself --------------------------------------------------------------------------------
@pytest.mark.parametrize("mirror", [True, False])
def test_exact_reference_matches_oracle(mirror):
    """exact_sums / expected_ll_mse on a small integer problem against orc.elbo_parts and orc.reconstruction_mse"""
    n, T, r = 11, 5, 2
    c = int_constants(n, T, r)
    Xm, Xc = int_state(n, T, r, seed=1, structure="good", device="cpu")
    Y = int_Y(Xm, r, seed=2, mirror=mirror, chunk=4)
    Ynp = Y.numpy()
    offd = ~np.eye(n, dtype=bool)
    assert mirror == np.array_equal(Ynp[offd][:, :, 0], np.swapaxes(Ynp, 0, 1)[offd][:, :, 1])
    assert np.all(np.abs(Ynp[offd]) <= 4 + 4 * r + 3)
    s = exact_sums(Y, Xm, Xc, r, chunk=4)
    s1 = exact_sums(Y, Xm, Xc, r, chunk=64)
    assert s == s1
    xm, xc = Xm.numpy(), Xc.numpy()
    for mode in (orc.NAIVE, orc.GOOD):
        lls, mse = expected_ll_mse(s, n, T, c["d"], mode)
        ll, _, _, _ = orc.elbo_parts(Ynp, xm, xc, c, mode)
        assert abs(lls[0] - ll) <= 1e-12 * abs(ll), (mode, lls, ll)
        assert mse == orc.reconstruction_mse(Ynp, xm, c)
    # one residual moved by one: the integer sums move with it
    Y2 = Y.clone()
    Y2[3, 7, 2, 1] += 1
    s2 = exact_sums(Y2, Xm, Xc, r, chunk=4)
    assert s2["sq"] != s["sq"] and (s2["s11"], s2["s01"]) != (s["s11"], s["s01"])
