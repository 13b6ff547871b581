"""CPU replay of the shifted solves (H - z S) x = b (tests/emul/emul_shifted.cpp runs the device's per-thread bodies of
bsp_core.h and its step schedule on the host), against LAPACK (scipy.linalg.solve_banded, partial pivoting) and the
spectral sum C (C^T b) / (E - z), on the shapes tests/test_gpu_shifted.py runs on the device and with the same bars
(DESIGN.md section 9).  tests/test_gpu_shifted.py also compares device and replay bit for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.linalg import eigh, solve_banded

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "emul", "emul_shifted.cpp")
dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int)
EPS = np.finfo(float).eps
BERR_BAR = 64 * EPS          # BSP_SHIFT_BERR_BAR: above it a solved system reports info = n + 1
REL_LAPACK = 1e-10           # max |x - x_lapack| / max |x_lapack| for shifts >= 1e-4 (relative) from the spectrum
REL_SPECTRAL = 1e-9          # the same against C (C^T b) / (E - z) from all eigenpairs


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emul_shifted") / "libemul_shifted.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-o", so, SRC])
    lib = C.CDLL(so)
    lib.emul_shifted.argtypes = [C.c_int, C.c_int, dp, dp, dp, C.c_double, C.c_int, dp, C.c_int, C.c_int, dp, dp, ip, dp, ip]
    return lib


def upper_bands(A, B):
    n = A.shape[0]
    out = np.zeros((B + 1, n))
    for d in range(min(B, n - 1) + 1):
        out[d, :n - d] = np.diag(A, d)
    return out


def band_width(ka, kb, n):
    """the library's group half bandwidth (bspatom_band_upload)"""
    return max(min(max(ka, kb), n - 1), 2)


def replay(emul, H0, S, B, z, rhs, Q=None, cl=0.0):
    """rhs: (nsys, n, nrhs); returns X (NaN where not written), info, berr, corrections"""
    n = H0.shape[0]
    z = np.asarray(z)
    cplx = np.iscomplexobj(z) or np.iscomplexobj(rhs)
    dt = np.complex128 if cplx else np.float64
    nsys, nrhs = rhs.shape[0], rhs.shape[2]
    Bm = np.ascontiguousarray(np.transpose(rhs, (0, 2, 1)).astype(dt))       # per system: n x nrhs column-major
    X = np.full_like(Bm, np.nan)
    info, berr, steps = np.zeros(nsys, np.int32), np.zeros(nsys), C.c_int()
    zz = np.ascontiguousarray(z.astype(dt))
    h0b, sb = upper_bands(H0, B), upper_bands(S, B)
    qb = upper_bands(Q, B) if Q is not None else np.zeros_like(h0b)
    rc = emul.emul_shifted(n, B, h0b.ctypes.data_as(dp), qb.ctypes.data_as(dp), sb.ctypes.data_as(dp), cl, nsys,
                           zz.ctypes.data_as(dp), nrhs, int(cplx), Bm.ctypes.data_as(dp), X.ctypes.data_as(dp),
                           info.ctypes.data_as(ip), berr.ctypes.data_as(dp), C.byref(steps))
    assert rc == 0
    return np.transpose(X, (0, 2, 1)), info, berr, steps.value


def lapack_solve(H, S, z, b, kd):
    M = H - z * S
    n = M.shape[0]
    ab = np.zeros((2 * kd + 1, n), dtype=M.dtype)
    for d in range(-kd, kd + 1):
        if d >= 0:
            ab[kd - d, d:] = np.diag(M, d)
        else:
            ab[kd - d, :d] = np.diag(M, d)
    return solve_banded((kd, kd), ab, np.asarray(b, dtype=M.dtype))


def rel_err(x, ref):
    return np.abs(x - ref).max() / np.abs(ref).max()


def shifts_across(w, count, rng, rel=1e-4, top=5.0):
    """real shifts spread over the spectrum (below its bottom to `top`), at least rel (relative) from every eigenvalue"""
    out = []
    lo, hi = w[0] - 0.2 * abs(w[0]), min(w[-1], top)
    while len(out) < count:
        z = rng.uniform(lo, hi)
        if np.min(np.abs(w - z)) > rel * max(abs(z), 1e-2):
            out.append(z)
    return np.array(out)


@pytest.fixture(scope="module")
def cfg2():
    from oracle import oracle as O

    b = O.make_basis(kind_grid=0, k=7, nfun=1000, rb=500.0)
    m = O.matrix_svt(b, lmax=50, par=O.pot_params(0, 1.0))
    pens = {}
    for l in (0, 1, 17, 50):
        H = O.hamiltonian(m["T"], m["U"][:, :, l], m["V"])
        w, Cv = eigh(H, m["S"])
        pens[l] = (H, w, Cv)
    return O, b, m, pens


@pytest.mark.parametrize("l", [0, 1, 17, 50])
@pytest.mark.parametrize("kind", ["real", "complex"])
def test_cfg2_shifts_against_lapack_and_spectral_sum(emul, cfg2, l, kind):
    O, b, m, pens = cfg2
    H, w, Cv = pens[l]
    S, n = m["S"], b.nfun
    rng = np.random.default_rng(100 + l + (kind == "complex"))
    if kind == "real":
        z = shifts_across(w, 8, rng)
    else:    # z = E_1s + omega + i eta with omega above threshold
        z = w[0] + np.abs(w[0]) + rng.uniform(0.05, 2.0, 8) + 1j * np.array([1e-3, 1e-1] * 4)
    rhs = rng.standard_normal((len(z), n, 2)) * np.exp(-np.linspace(0.0, 25.0, n))[None, :, None]
    X, info, berr, steps = replay(emul, H, S, 6, z, rhs)
    assert np.all(info == 0) and np.all(berr <= BERR_BAR), (info, berr)
    assert 1 <= steps <= 5
    for s in range(len(z)):
        for c in range(2):
            ref = lapack_solve(H, S, z[s], rhs[s, :, c], 6)
            assert rel_err(X[s, :, c], ref) <= REL_LAPACK
            spec = Cv @ ((Cv.T @ rhs[s, :, c]) / (w - z[s]))
            assert rel_err(X[s, :, c], spec) <= REL_SPECTRAL


def test_hydrogen_static_polarisability(emul, cfg2):
    """alpha(0) = 2/3 b^T x, (H_1 - E_1s S) x = b, b = R c_1s: 9/2 for hydrogen"""
    O, b, m, pens = cfg2
    w0, C0 = pens[0][1], pens[0][2]
    bvec = m["R"] @ C0[:, 0]
    X, info, berr, _ = replay(emul, pens[1][0], m["S"], 6, [w0[0]], bvec[None, :, None])
    assert info[0] == 0
    alpha = 2.0 / 3.0 * bvec @ X[0, :, 0]
    assert abs(alpha - 4.5) < 1e-8, alpha


def fem_hydrogen(nel, p, R):
    """radial hydrogen (l = 0), Lagrange elements of degree p on [0, R]: stiffness / 2 - 1/r and the mass matrix"""
    xg, wg = np.polynomial.legendre.leggauss(p + 6)
    t, wt = (xg + 1) / 2, wg / 2
    nodes = np.linspace(0.0, 1.0, p + 1)
    coef = np.linalg.inv(np.vander(nodes, p + 1, increasing=True))
    powers = np.vander(t, p + 1, increasing=True)
    dpowers = np.hstack([np.zeros((len(t), 1)), powers[:, :-1] * np.arange(1, p + 1)])
    phi, dphi = (powers @ coef).T, (dpowers @ coef).T
    h = R / nel
    nn = nel * p + 1
    A, B = np.zeros((nn, nn)), np.zeros((nn, nn))
    for e in range(nel):
        r = (e + t) * h
        ix = np.ix_(e * p + np.arange(p + 1), e * p + np.arange(p + 1))
        wq = wt * h
        B[ix] += (phi * wq) @ phi.T
        A[ix] += 0.5 * ((dphi / h) * wq) @ (dphi / h).T - (phi * (wq / r)) @ phi.T
    return A[1:-1, 1:-1], B[1:-1, 1:-1]


def random_pencil(rng, n, ka, kb):
    A, B = np.zeros((n, n)), np.zeros((n, n))
    for d in range(min(ka, n - 1) + 1):
        v = rng.uniform(-1, 1, n - d)
        A += np.diag(v, d) + (np.diag(v, -d) if d else 0)
    for d in range(1, min(kb, n - 1) + 1):
        v = rng.uniform(-0.5, 0.5, n - d)
        B += np.diag(v, d) + np.diag(v, -d)
    B += np.diag(np.abs(B).sum(1) + rng.uniform(0.5, 1.5, n))
    return A, B


def band_cases():
    rng = np.random.default_rng(20261022)
    out = [("fem1", *fem_hydrogen(2000, 1, 60.0), 1, 1), ("fem1 n=4000", *fem_hydrogen(4001, 1, 80.0), 1, 1),
           ("fem1 n=1", *fem_hydrogen(2, 1, 10.0), 1, 1)]
    for n, ka, kb in ((2, 1, 2), (6, 5, 2), (300, 9, 4), (500, 2, 7), (200, 0, 3)):
        out.append(("random n=%d" % n, *random_pencil(rng, n, ka, kb), ka, kb))
    return out


@pytest.mark.parametrize("case", range(8))
def test_band_pencils_against_lapack(emul, case):
    name, A, Bm, ka, kb = band_cases()[case]
    n = A.shape[0]
    kd = band_width(ka, kb, n)
    w = eigh(A, Bm, eigvals_only=True)
    rng = np.random.default_rng(case)
    z = np.r_[shifts_across(w, 3, rng, top=w[-1]), w[0] + 0.3 + 0.05j]
    rhs = rng.standard_normal((len(z), n, 1))
    for zz in (z[:3], z[3:]):
        X, info, berr, _ = replay(emul, A, Bm, kd, zz, rhs[:len(zz)])
        assert np.all(info == 0) and np.all(berr <= BERR_BAR), (name, info, berr)
        for s in range(len(zz)):
            assert rel_err(X[s, :, 0], lapack_solve(A, Bm, zz[s], rhs[s, :, 0], max(ka, kb))) <= REL_LAPACK, name


@pytest.mark.parametrize("nrhs", [0, 1, 3, 9])
def test_right_hand_side_counts(emul, cfg2, nrhs):
    O, b, m, pens = cfg2
    H, w, _ = pens[17]
    rng = np.random.default_rng(nrhs)
    z = shifts_across(w, 3, rng)
    rhs = rng.standard_normal((3, b.nfun, nrhs))
    X, info, berr, _ = replay(emul, H, m["S"], 6, z, rhs)
    assert np.all(info == 0) and np.all(berr <= BERR_BAR)
    for s in range(3):
        for c in range(nrhs):
            assert rel_err(X[s, :, c], lapack_solve(H, m["S"], z[s], rhs[s, :, c], 6)) <= REL_LAPACK
        # every column is its own refinement: solved alone it gives the same bits
        for c in range(nrhs):
            Xc, *_ = replay(emul, H, m["S"], 6, z[s:s + 1], rhs[s:s + 1, :, c:c + 1])
            assert np.array_equal(Xc[0, :, 0].view(np.int64), X[s, :, c].view(np.int64))


def test_zero_first_pivot(emul):
    A, Bm = np.array([[0.0, 1.0], [1.0, 0.0]]), np.eye(2)
    X, info, berr, _ = replay(emul, A, Bm, 2, [0.0, 0.5], np.ones((2, 2, 1)))
    assert info[0] == 1 and np.all(np.isnan(X[0]))
    assert info[1] == 0
    assert np.allclose(X[1, :, 0], np.linalg.solve(A - 0.5 * Bm, np.ones(2)), rtol=1e-14)


def test_shift_at_a_computed_eigenvalue(emul, cfg2):
    """info says what happened: n + 1 exactly when berr is above the bar, and X is finite unless a pivot failed"""
    O, b, m, pens = cfg2
    H, w, _ = pens[0]
    z = w[[0, 5, 400]]
    X, info, berr, _ = replay(emul, H, m["S"], 6, z, np.ones((3, b.nfun, 1)))
    for s in range(3):
        if 1 <= info[s] <= b.nfun:
            continue
        assert (info[s] == b.nfun + 1) == (berr[s] > BERR_BAR)
        assert np.all(np.isfinite(X[s]))


def test_non_finite_right_hand_side_is_reported(emul, cfg2):
    """a NaN or Inf in b makes the backward error NaN: the column is reported (info = n + 1), not solved"""
    O, b, m, pens = cfg2
    H, w, _ = pens[1]
    rhs = np.ones((3, b.nfun, 2))
    rhs[0, 17, 0] = np.nan
    rhs[1, 400, 1] = np.inf
    X, info, berr, _ = replay(emul, H, m["S"], 6, [0.1, 0.1, 0.1], rhs)
    assert list(info) == [b.nfun + 1, b.nfun + 1, 0]
    assert np.isnan(berr[0]) and np.isnan(berr[1]) and berr[2] <= BERR_BAR
