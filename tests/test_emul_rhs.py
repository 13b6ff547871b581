"""The factor sweep forms its own right-hand side from the vector in X: S x for the second solve, (H - rho S) x for a
correction.  These values used to be summed by the back sweep's column sweep (and by a separate residual pass) and
written to HBM; the solver's results stay bit for bit the same only if the factor sweep sums in exactly that order.

CPU replay (tests/emul/emul_rhs.cpp) of bsp_factor_forward_rows on cfg2-shaped pencils (N = 1000 B-splines of order
7 on the linear grid, Rmax = 500, Coulomb), compared with the column-sweep order bit for bit.  A deliberately wrong
order must be caught."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "emul", "emul_rhs.cpp")
dp = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emul_rhs") / "libemul_rhs.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-o", so, SRC])
    lib = C.CDLL(so)
    lib.emul_rhs.argtypes = [C.c_int, C.c_int, dp, dp, dp, C.c_double, C.c_int, C.c_int, dp, dp]
    return lib


@pytest.fixture(scope="module")
def cfg2_matrices():
    from oracle import oracle as O

    b = O.make_basis(kind_grid=0, k=7, nfun=1000, rb=500.0)
    assert b.nfun == 1000
    return O, b, O.matrix_svt(b, lmax=50, par=O.pot_params(0, 1.0 + 5 / 64.0))


def upper_bands(A, B):
    n = A.shape[0]
    return np.ascontiguousarray(np.stack([np.r_[np.diag(A, d), np.zeros(d)] for d in range(B + 1)]))


def formed_and_reference(emul, H, S, B, x, rho, resid, swap=0):
    n = len(x)
    hb, sb = upper_bands(H, B), upper_bands(S, B)
    x = np.ascontiguousarray(x, dtype=np.float64)
    fused, ref = np.empty(n), np.empty(n)
    rc = emul.emul_rhs(n, B, hb.ctypes.data_as(dp), sb.ctypes.data_as(dp), x.ctypes.data_as(dp), rho, resid, swap,
                       fused.ctypes.data_as(dp), ref.ctypes.data_as(dp))
    assert rc == 0
    seen = ~np.isnan(fused)
    return fused, ref, seen


@pytest.mark.parametrize("l", [0, 1, 17, 50])
@pytest.mark.parametrize("resid", [0, 1], ids=["Sx", "H-rhoS"])
def test_formed_rhs_matches_column_sweep_bits_cfg2(emul, cfg2_matrices, l, resid):
    O, b, m = cfg2_matrices
    H = O.hamiltonian(m["T"], m["U"][:, :, l], m["V"])
    S = m["S"]
    B = b.k - 1
    rng = np.random.default_rng(1000 + 7 * l + resid)
    n = b.nfun
    # a vector with the spread of magnitudes of a bound state, and a random one
    for x in (np.exp(-np.linspace(0.0, 30.0, n)) * rng.standard_normal(n), rng.uniform(-1.0, 1.0, n)):
        rho = float(np.dot(x, H @ x) / np.dot(x, S @ x)) if resid else 0.0
        fused, ref, seen = formed_and_reference(emul, H, S, B, x, rho, resid)
        # the check-points hold rows js+7 .. js+13 of every 14-row segment: half of all rows, in every position
        assert seen.sum() >= n // 2 - 7
        assert np.array_equal(fused[seen].view(np.int64), ref[seen].view(np.int64))
        # the values are what they should be: the band matvec
        want = (H @ x - rho * (S @ x)) if resid else S @ x
        scale = np.abs(H).max() * np.abs(x).max() + np.abs(rho) * np.abs(S).max() * np.abs(x).max()
        assert np.abs(ref - want).max() <= 64 * np.finfo(float).eps * scale


@pytest.mark.parametrize("resid", [0, 1], ids=["Sx", "H-rhoS"])
def test_wrong_summation_order_is_caught(emul, cfg2_matrices, resid):
    O, b, m = cfg2_matrices
    H = O.hamiltonian(m["T"], m["U"][:, :, 50], m["V"])
    x = np.random.default_rng(7).uniform(-1.0, 1.0, b.nfun)
    rho = 0.37 if resid else 0.0
    fused, ref, seen = formed_and_reference(emul, H, m["S"], b.k - 1, x, rho, resid, swap=1)
    assert not np.array_equal(fused[seen].view(np.int64), ref[seen].view(np.int64))


@pytest.mark.parametrize("k,n", [(2, 37), (5, 64), (8, 200), (10, 101)])
def test_formed_rhs_other_band_widths(emul, k, n):
    """short and wide bands, and sizes that leave a partial last segment"""
    from oracle import oracle as O

    b = O.make_basis(kind_grid=0, k=k, nfun=n, rb=40.0)
    m = O.matrix_svt(b, lmax=2, par=O.pot_params(0, 2.0))
    H = O.hamiltonian(m["T"], m["U"][:, :, 2], m["V"])
    x = np.random.default_rng(k * 1000 + n).standard_normal(b.nfun)
    for resid in (0, 1):
        fused, ref, seen = formed_and_reference(emul, H, m["S"], k - 1, x, -0.5 if resid else 0.0, resid)
        assert seen.any()
        assert np.array_equal(fused[seen].view(np.int64), ref[seen].view(np.int64))
