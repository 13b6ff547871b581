"""GPU: caller-supplied band pencils (bspatom_band_upload / bspatom_solve_band_batch / bspatom_dsbgv_, DSBGV semantics).

The band front end only replaces the assembly: it writes the full-band rows the solver reads.  So the library's own
B-spline bands, handed back in as band pencils, must give the assembled path's bits exactly (at l > 0 with
H_l = fma(l(l+1), Q, H0) rounded once, which is what bsp_combine_kernel computes), on every delivery path.  Pencils that
are not B-splines (linear and cubic FEM hydrogen, seeded random pencils) are checked against LAPACK on the dense
pencil."""
import ctypes as C
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest
from scipy.linalg import eigh, lapack

import bspatom_b200 as bsp
from bspatom_b200 import _lib
from bspatom_b200.host import pinned_empty
from cases import band_to_dense_general, check_eigenpairs, eig_tolerance, host_basis

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 1000
ZS = [1.0, 1.0 + 1 / 64.0, 1.5]


def cfg2_basis(grid):
    if grid == "lin":
        a = host_basis(kind_grid=0, k=7, nfun=N, rb=500.0)
    else:
        a = host_basis(kind_grid=2, k=7, nfun=782, rb=500.0, rmax=70.0)
    assert a.nfun == N
    return a


def coulomb(a, z):
    return bsp.Problem(k=a.k, nfun=a.nfun, nkp=a.nkp, ka=a.ka, rt=a.rt, pot_kind=bsp.POT_COULOMB, pot_par=(z,))


def to_lower(ab):
    """LAPACK upper band (kd+1, n) -> lower band storage of the same symmetric matrix: L[r, j] = A(j+r, j)"""
    kd, n = ab.shape[0] - 1, ab.shape[1]
    lo = np.zeros_like(ab, order="F")
    for r in range(kd + 1):
        lo[r, :n - r] = ab[kd - r, r:]
    return lo


def dense_to_upper(A, kd):
    n = A.shape[0]
    ab = np.zeros((kd + 1, n), order="F")
    for d in range(kd + 1):
        ab[kd - d, d:] = np.diagonal(A, d)
    return ab


def fma_rounded(c, Q, H0):
    """fma(c, Q, H0) entrywise with one rounding (exact in rationals, then float)"""
    fc = Fraction(c)
    out = [float(fc * Fraction(float(q)) + Fraction(float(h))) for q, h in zip(Q.ravel(), H0.ravel())]
    return np.asfortranarray(np.reshape(out, H0.shape))


def assert_bits(a, b):
    assert np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64))


def assert_same_result(got, ref):
    (E1, C1, i1), (E2, C2, i2) = got, ref
    assert np.array_equal(i1, i2)
    for x, y in zip(E1, E2):
        assert_bits(x, y)
    for x, y in zip(C1, C2):
        assert_bits(x, y)


# ---- bit identity with the assembled path -------------------------------------------------------------------------
@pytest.mark.parametrize("grid", ["lin", "explin"])
def test_l0_band_pencils_give_the_assembled_bits(atom, grid):
    a = cfg2_basis(grid)
    probs = [coulomb(a, z) for z in ZS]
    ref = atom.solve_batch([(p, 0) for p in probs])
    assert not ref[2].any()
    bands = [atom.MATRIX_SVT(p) for p in probs]
    up = [(b["H0"], b["S"]) for b in bands]
    lo = [(to_lower(b["H0"]), to_lower(b["S"]), "L") for b in bands]
    for pens in (up, lo):
        assert_same_result(atom.solve_band_batch(pens), ref)


@pytest.mark.parametrize("l", [1, 17, 50])
def test_l_positive_with_host_formed_h_gives_the_assembled_bits(atom, l):
    a = cfg2_basis("lin")
    probs = [coulomb(a, z) for z in ZS[:2]]
    ref = atom.solve_batch([(p, l) for p in probs])
    assert not ref[2].any()
    pens = []
    for p in probs:
        b = atom.MATRIX_SVT(p)
        pens.append((fma_rounded(float(l * (l + 1)), b["Q"], b["H0"]), b["S"]))
    assert_same_result(atom.solve_band_batch(pens), ref)


# ---- the full cfg2 step through every delivery path -----------------------------------------------------------------
def cfg2_step_pencils(atom):
    """408 pencils: l = 0..50 x 8 charges, S and H_l = H0 + l(l+1) Q from bspatom_assemble_band"""
    a = cfg2_basis("lin")
    pens = []
    for i in range(8):
        b = atom.MATRIX_SVT(coulomb(a, 1.0 + i / 64.0))
        pens += [(np.asfortranarray(b["H0"] + (l * (l + 1)) * b["Q"]), b["S"]) for l in range(51)]
    return pens


def test_full_step_resident_streamed_and_redone_agree(atom):
    pens = cfg2_step_pencils(atom)
    npen = len(pens)
    assert npen == 408
    atom.band_upload(pens)
    atom.batch_run()
    E, Cb, info = np.full(npen * N, np.nan), np.full(npen * N * N, np.nan), np.full(npen, -1, np.int32)
    atom.batch_download(E, Cb, info)
    assert not info.any()
    v = atom.batch_verify()
    assert v["max_scaled_residual"] <= 1e-11 and v["max_orthonormality_defect"] <= 1e-9
    assert v["not_ascending"] == 0.0 and v["eigenpairs_checked"] == npen * N
    pE, pC = pinned_empty(npen * N), pinned_empty(npen * N * N)

    def streamed():
        pE.fill(np.nan)
        pC.fill(np.nan)
        _, _, inf = atom.solve_band_batch(pens, out_E=pE, out_C=pC)
        assert np.array_equal(inf, info)
        assert_bits(pE, E)
        assert_bits(pC, Cb)

    streamed()
    atom.set_option("rounds_enqueued", 1)
    try:
        atom.band_upload(pens)
        atom.batch_run()
        assert atom.stats()["chunks_redone"] >= 1
        E2, C2, i2 = np.full(npen * N, np.nan), np.full(npen * N * N, np.nan), np.full(npen, -1, np.int32)
        atom.batch_download(E2, C2, i2)
        assert np.array_equal(i2, info)
        assert_bits(E2, E)
        assert_bits(C2, Cb)
        streamed()
        assert atom.stats()["chunks_redone"] >= 1
    finally:
        atom.set_option("rounds_enqueued", 26)


# ---- pencils that are not B-splines, against LAPACK -----------------------------------------------------------------
def fem_hydrogen(nel, p, R):
    """radial hydrogen (l = 0) with Lagrange elements of degree p on [0, R], psi(0) = psi(R) = 0: stiffness / 2 - 1/r
    and the consistent mass matrix, dense, half bandwidth p"""
    xg, wg = np.polynomial.legendre.leggauss(p + 6)
    t, wt = (xg + 1) / 2, wg / 2
    nodes = np.linspace(0.0, 1.0, p + 1)
    coef = np.linalg.inv(np.vander(nodes, p + 1, increasing=True))      # phi_a(t) = sum_k coef[k, a] t^k
    powers = np.vander(t, p + 1, increasing=True)
    dpowers = np.hstack([np.zeros((len(t), 1)), powers[:, :-1] * np.arange(1, p + 1)])
    phi, dphi = (powers @ coef).T, (dpowers @ coef).T
    h = R / nel
    nn = nel * p + 1
    A, B = np.zeros((nn, nn)), np.zeros((nn, nn))
    for e in range(nel):
        r = (e + t) * h
        ix = np.ix_(e * p + np.arange(p + 1), e * p + np.arange(p + 1))
        w = wt * h
        B[ix] += (phi * w) @ phi.T
        A[ix] += 0.5 * ((dphi / h) * w) @ (dphi / h).T - (phi * (w / r)) @ phi.T
    return A[1:-1, 1:-1], B[1:-1, 1:-1]


def random_pencil(rng, n, ka, kb):
    """symmetric A with half bandwidth ka, symmetric positive definite B (diagonally dominant) with half bandwidth kb"""
    A, B = np.zeros((n, n)), np.zeros((n, n))
    for d in range(min(ka, n - 1) + 1):
        v = rng.uniform(-1, 1, n - d)
        A += np.diag(v, d) + (np.diag(v, -d) if d else 0)
    for d in range(1, min(kb, n - 1) + 1):
        v = rng.uniform(-0.5, 0.5, n - d)
        B += np.diag(v, d) + np.diag(v, -d)
    B += np.diag(np.abs(B).sum(1) + rng.uniform(0.5, 1.5, n))
    return A, B


def store(M, k, uplo, ld=None):
    """dense symmetric -> LAPACK band storage with leading dimension ld (a Fortran view into a taller buffer)"""
    ab = dense_to_upper(M, k) if uplo == "U" else to_lower(dense_to_upper(M, k))
    if ld is None or ld == k + 1:
        return ab
    buf = np.full((ld, M.shape[0]), 7.0, order="F")     # rows beyond k + 1 are never read
    buf[:k + 1] = ab
    return buf[:k + 1]


def non_bspline_cases():
    rng = np.random.default_rng(20261020)
    cases = []   # (name, A, B, ka, kb, uplo, ld extra, nvec)
    A, B = fem_hydrogen(2000, 1, 60.0)
    cases.append(("fem1 hydrogen", A, B, 1, 1, "U", 0, A.shape[0] // 3))
    A, B = fem_hydrogen(700, 3, 60.0)
    cases.append(("fem3 hydrogen", A, B, 3, 3, "L", 0, A.shape[0] // 3))
    A, B = fem_hydrogen(4001, 1, 80.0)
    cases.append(("fem1 n=4000", A, B, 1, 1, "L", 2, 1))
    A, B = fem_hydrogen(2, 1, 10.0)
    cases.append(("fem1 n=1", A, B, 1, 1, "U", 0, 1))
    A, B = fem_hydrogen(1, 3, 10.0)
    cases.append(("fem3 n=2", A, B, 3, 3, "U", 0, 2))
    for n, ka, kb, uplo, extra, nv in ((1, 2, 0, "L", 1, 1), (2, 1, 2, "U", 0, 0), (6, 5, 2, "U", 3, 6), (4, 3, 1, "L", 0, 1),
                                       (300, 9, 4, "U", 3, 100), (500, 2, 7, "L", 1, 500), (200, 0, 3, "U", 0, 0),
                                       (300, 4, 9, "L", 2, 300)):
        A, B = random_pencil(rng, n, ka, kb)
        w = eigh(A, B, eigvals_only=True)
        if n > 1:     # relative gaps far above rounding: each eigenvector is determined to ~eps / gap << 1e-9
            assert np.diff(w).min() > 1e-6 * np.abs(w).max(), (n, ka, kb, np.diff(w).min())
        cases.append(("random n=%d ka=%d kb=%d" % (n, ka, kb), A, B, ka, kb, uplo, extra, nv))
    return cases


def test_non_bspline_pencils_match_lapack_in_one_mixed_batch(atom, oracle):
    cases = non_bspline_cases()
    pens, nvecs = [], []
    for _, A, B, ka, kb, uplo, extra, nv in cases:
        pens.append((store(A, ka, uplo, ka + 1 + extra), store(B, kb, uplo, kb + 1 + extra), uplo))
        nvecs.append(nv)
    assert any(p[0].strides[1] > 8 * p[0].shape[0] for p in pens)
    Es, Cs, info = atom.solve_band_batch(pens, nvec=nvecs)
    assert not info.any(), info
    for (name, A, B, ka, kb, uplo, extra, nv), E, Cm in zip(cases, Es, Cs):
        w, _, inf = oracle.dsygv(A, B)
        assert inf == 0
        assert np.all(np.abs(E - w) <= eig_tolerance(w)), name
        assert Cm.shape == (A.shape[0], nv)
        if nv:
            check_eigenpairs(E, Cm, A, B, res_tol=1e-11, orth_tol=1e-9)
        if name.endswith("hydrogen"):
            assert np.all(np.abs(E[:3] + 0.5 / np.arange(1, 4) ** 2) <= 2e-3), (name, E[:3])


# ---- input the Python layer has to copy; many pencils of one shape --------------------------------------------------
def test_copied_operands_give_the_bits_of_fortran_input(atom):
    """C-ordered operands are copied into Fortran order by the Python layer: the copies must live through the C call
    (band_upload and solve_band_batch), so the results equal those of Fortran-ordered input bit for bit"""
    rng = np.random.default_rng(23)
    pen = [random_pencil(rng, 300, 4, 2) for _ in range(3)]
    fort = [(dense_to_upper(A, 4), dense_to_upper(B, 2)) for A, B in pen]
    ref = atom.solve_band_batch(fort)
    assert not ref[2].any()

    def c_ordered():
        return [(np.ascontiguousarray(a), np.ascontiguousarray(b)) for a, b in fort]

    assert_same_result(atom.solve_band_batch(c_ordered()), ref)
    atom.band_upload(c_ordered())
    junk = [np.full((5, 300), 123.0) for _ in range(64)]      # reuse any freed host block before the run
    atom.batch_run()
    E, Cb, info = np.zeros(900), np.zeros(3 * 300 * 300), np.full(3, -1, np.int32)
    atom.batch_download(E, Cb, info)
    del junk
    assert_same_result(([E[i * 300:(i + 1) * 300] for i in range(3)],
                        [Cb[i * 90000:(i + 1) * 90000].reshape((300, 300), order="F") for i in range(3)], info), ref)


def test_more_pencils_of_one_shape_than_a_grid_dimension_holds(atom):
    """70 000 pencils of one (n, B) group: more than the 65 535 blocks a launch has along y"""
    rng = np.random.default_rng(29)
    A, B = random_pencil(rng, 5, 1, 1)
    ab, bb = dense_to_upper(A, 1), dense_to_upper(B, 1)
    one = atom.solve_band_batch([(ab, bb)], nvec=1)
    Es, Cs, info = atom.solve_band_batch([(ab, bb)] * 70000, nvec=1)
    assert not info.any()
    assert np.array_equal(np.concatenate(Es), np.tile(one[0][0], 70000))
    assert np.array_equal(np.concatenate([c.ravel() for c in Cs]), np.tile(one[1][0].ravel(), 70000))
    w = eigh(A, B, eigvals_only=True)
    assert np.all(np.abs(one[0][0] - w) <= eig_tolerance(w))


# ---- errors -----------------------------------------------------------------------------------------------------------
def small_valid():
    rng = np.random.default_rng(5)
    A, B = random_pencil(rng, 40, 2, 1)
    return [(dense_to_upper(A, 2), dense_to_upper(B, 1)), (dense_to_upper(A, 2), dense_to_upper(B, 1))], A, B


def raw_solve(atom, arr, n):
    E, Cb, info = np.zeros(n * 40), np.zeros(n * 40 * 40), np.zeros(n, np.int32)
    return atom.lib.bspatom_solve_band_batch(atom._h, n, arr, E.ctypes.data_as(C.c_void_p), Cb.ctypes.data_as(C.c_void_p),
                                             info.ctypes.data_as(C.c_void_p))


def test_errors_leave_the_handle_usable(atom):
    pens, A, B = small_valid()
    ref = atom.solve_band_batch(pens)
    assert not ref[2].any()
    wide = np.zeros((11, 40), order="F")
    wide[8:] = pens[0][0]

    def broken(edit):
        arr, keep, _, _ = bsp.host.band_pencil_array(pens)
        edit(arr[1], keep)
        return arr, keep

    bad = {
        "ka > 9": lambda p, k: (setattr(p, "ka", 10), setattr(p, "AB", wide.ctypes.data_as(_lib._dp)), setattr(p, "ldab", 11)),
        "kb > 9": lambda p, k: setattr(p, "kb", 10),
        "ldab": lambda p, k: setattr(p, "ldab", 2),
        "NULL BB": lambda p, k: setattr(p, "BB", None),
        "nvec < 0": lambda p, k: setattr(p, "nvec", -1),
        "nvec > n": lambda p, k: setattr(p, "nvec", 41),
        "uplo": lambda p, k: setattr(p, "uplo", b"X"),
    }
    for what, edit in bad.items():
        arr, keep = broken(edit)
        rc = raw_solve(atom, arr, 2)
        if what.startswith(("ka", "kb")):
            assert rc == _lib.EUNSUPPORTED, what
        else:
            assert rc < 0, what
        assert "index 1" in atom.lib.bspatom_last_error(atom._h).decode(), what
        assert_same_result(atom.solve_band_batch(pens), ref)


def test_nan_is_rejected_before_the_device_is_touched(atom):
    pens, A, B = small_valid()
    ref = atom.solve_band_batch(pens)
    nanA = pens[1][0].copy(order="F")
    nanA[2, 7] = np.nan                                       # stored diagonal
    with pytest.raises(bsp.BspAtomError, match="index 1.*AB"):
        atom.band_upload([pens[0], (nanA, pens[1][1])])
    # the resident batch of the last call is still there: nothing was freed or uploaded
    E, Cb, info = np.zeros(80), np.zeros(2 * 1600), np.full(2, -1, np.int32)
    atom.batch_download(E, Cb, info)
    assert_bits(E, np.concatenate(ref[0]))
    assert_bits(Cb, np.concatenate([c.ravel(order="F") for c in ref[1]]))
    # a NaN outside the stored triangle (upper storage, column 0, rows 0..ka-1) is never read
    corner = pens[1][0].copy(order="F")
    corner[0, 0] = np.nan
    assert_same_result(atom.solve_band_batch([pens[0], (corner, pens[1][1])]), ref)


# ---- B not positive definite; a degenerate pencil ---------------------------------------------------------------------
def test_indefinite_b_is_reported_and_leaves_its_slots_alone(atom):
    rng = np.random.default_rng(11)
    n, i_bad = 120, 37
    pen = [random_pencil(rng, n, 3, 2) for _ in range(3)]
    Bbad = pen[1][1].copy()
    Bbad[i_bad - 1, i_bad - 1] = -1.0
    bb = dense_to_upper(Bbad, 2)
    _, pinfo = lapack.dpbtrf(bb, lower=0)
    assert pinfo == i_bad
    pens = [(dense_to_upper(A, 3), dense_to_upper(B, 2)) for A, B in pen]
    good = atom.solve_band_batch([pens[0], pens[2]])
    E, Cb = pinned_empty(3 * n), pinned_empty(3 * n * n)
    E.fill(12345.0)
    Cb.fill(12345.0)
    Es, Cs, info = atom.solve_band_batch([pens[0], (pens[1][0], bb), pens[2]], out_E=E, out_C=Cb)
    assert list(info) == [0, n + i_bad, 0]
    assert np.all(Es[1] == 12345.0) and np.all(Cs[1] == 12345.0)
    assert_same_result(([Es[0], Es[2]], [Cs[0], Cs[2]], info[[0, 2]]), good)
    # the same pencil through the staged path
    atom.band_upload([pens[0], (pens[1][0], bb), pens[2]])
    atom.batch_run()
    E2, C2, i2 = np.full(3 * n, 7.0), np.full(3 * n * n, 7.0), np.full(3, -1, np.int32)
    atom.batch_download(E2, C2, i2)
    assert list(i2) == [0, n + i_bad, 0] and np.all(E2[n:2 * n] == 7.0)
    assert list(atom.selection()) == [n, 0, n]


def test_degenerate_pencil_is_reported(atom):
    rng = np.random.default_rng(3)
    A1, B1 = random_pencil(rng, 50, 2, 1)
    Z = np.zeros((50, 50))
    A, B = np.block([[A1, Z], [Z, A1]]), np.block([[B1, Z], [Z, B1]])
    others = [random_pencil(rng, 80, 2, 1) for _ in range(2)]
    pens = [(dense_to_upper(a, 2), dense_to_upper(b, 1)) for a, b in others]
    ref = atom.solve_band_batch(pens)
    assert not ref[2].any()
    Es, Cs, info = atom.solve_band_batch([pens[0], (dense_to_upper(A, 2), dense_to_upper(B, 1)), pens[1]])
    assert info[1] > 0 and info[0] == 0 and info[2] == 0
    assert_same_result(([Es[0], Es[2]], [Cs[0], Cs[2]], info[[0, 2]]), ref)


# ---- what the resident batch supports afterwards -------------------------------------------------------------------
def test_state_after_a_band_batch(atom):
    rng = np.random.default_rng(9)
    n, nl, nv = 150, 4, 30
    pen = [random_pencil(rng, n, 3, 3) for _ in range(nl)]
    pens = [(dense_to_upper(A, 3), dense_to_upper(B, 3)) for A, B in pen]
    atom.band_upload(pens, nvec=nv)
    atom.batch_run()
    E, Cb, info = np.zeros(nl * n), np.zeros(nl * n * nv), np.zeros(nl, np.int32)
    atom.batch_download(E, Cb, info)
    assert not info.any()
    with pytest.raises(bsp.BspAtomError, match="rc=1004"):
        atom.wavefunction_resident(0, 0, 1, 0.0, 1.0, npts=10)
    kd = 2
    Ab = np.asfortranarray(rng.uniform(-1, 1, (2 * kd + 1, n)))
    D = atom.dipole_chain_resident(Ab, 0, nl, nv)
    Ad = band_to_dense_general(Ab, n)
    Cl = [Cb[i * n * nv:(i + 1) * n * nv].reshape((n, nv), order="F") for i in range(nl)]
    for l in range(nl - 1):
        want = Cl[l + 1].T @ Ad @ Cl[l]
        assert np.abs(D[l] - want).max() <= 1e-12 * max(1.0, np.abs(want).max())
    # an assembled batch next on the same handle: the bits of a fresh handle
    a = host_basis(kind_grid=0, k=7, nfun=200, rb=100.0)
    items = [(a.problem(), l) for l in range(3)]
    got = atom.solve_batch(items, nvec=20)
    fresh = bsp.BspAtom(device=0)
    try:
        assert_same_result(got, fresh.solve_batch(items, nvec=20))
    finally:
        fresh.close()


# ---- bsp.dsbgv ----------------------------------------------------------------------------------------------------------
def test_dsbgv(atom, oracle):
    rng = np.random.default_rng(17)
    A, B = random_pencil(rng, 90, 4, 2)
    for uplo in "UL":
        ab, bb = store(A, 4, uplo), store(B, 2, uplo)
        ab0, bb0 = ab.copy(), bb.copy()
        w, Z, info = bsp.dsbgv(ab, bb, uplo=uplo)
        assert info == 0
        assert_bits(ab, ab0)
        assert_bits(bb, bb0)
        Es, Cs, inf = atom.solve_band_batch([(ab, bb, uplo)])
        assert_bits(w, Es[0])
        assert_bits(Z, Cs[0])
        wr, _, _ = oracle.dsygv(A, B)
        assert np.all(np.abs(w - wr) <= eig_tolerance(wr))
        check_eigenpairs(w, Z, A, B, res_tol=1e-11, orth_tol=1e-9)
        wn, Zn, info = bsp.dsbgv(ab, bb, jobz="N", uplo=uplo)
        assert info == 0 and Zn is None and np.all(np.abs(wn - wr) <= eig_tolerance(wr))
    ab, bb = store(A, 4, "U"), store(B, 2, "U")
    assert bsp.dsbgv(bb, ab)[2] == -5                       # kb > ka
    assert bsp.dsbgv(ab, bb, jobz="X")[2] == -1
    assert bsp.dsbgv(ab, bb, uplo="X")[2] == -2
    assert bsp.dsbgv(np.zeros((11, 90), order="F"), bb)[2] == -4
    Bbad = B.copy()
    Bbad[4, 4] = -1.0
    assert bsp.dsbgv(ab, store(Bbad, 2, "U"))[2] == 90 + 5


# ---- a C program through the header alone ---------------------------------------------------------------------------------
def test_c_band_driver(tmp_path):
    exe = str(tmp_path / "c_band_driver")
    libdir = os.path.join(ROOT, "bspatom_b200")
    subprocess.check_call(["gcc", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe,
                           os.path.join(ROOT, "tests", "c_band_driver.c"), "-L", libdir, "-lbspatom",
                           "-Wl,-rpath," + libdir, "-lm"])
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "c_band_driver: ok" in r.stdout, r.stdout + r.stderr
