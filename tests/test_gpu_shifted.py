"""GPU: the driven equation (A_p - z B_p) x = b on the resident batch (bspatom_shifted_solve[_z]).

Assembled cfg2 pencils (N = 1000, k = 7, l = 0, 1, 17, 50) and caller-supplied band pencils are solved for real shifts
spread over each spectrum and complex shifts above threshold, and checked against LAPACK (scipy.linalg.solve_banded)
on the library's own bands, against the spectral sum from the library's eigenpairs, against hydrogen's polarisability,
and bit for bit against the CPU replay of tests/emul/emul_shifted.cpp.  Bars: DESIGN.md section 9."""
import ctypes as C

import numpy as np
import pytest
from scipy.linalg import eigh

import bspatom_b200 as bsp
from bspatom_b200 import _lib
from cases import host_basis
from test_emul_shifted import (BERR_BAR, REL_LAPACK, band_width, emul, fem_hydrogen, lapack_solve, random_pencil,  # noqa: F401
                               rel_err, replay, shifts_across, upper_bands)

pytestmark = pytest.mark.gpu
LS = (0, 1, 17, 50)
REL_SPECTRAL_DEVICE = 1e-7   # against C (C^T b) / (E - z) from the library's eigenpairs (|C^T S C - I| <= 1e-9)


def bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def dense_from_upper(ab):
    kd, n = ab.shape[0] - 1, ab.shape[1]
    A = np.zeros((n, n))
    for d in range(kd + 1):
        v = ab[kd - d, d:]
        A += np.diag(v, d) + (np.diag(v, -d) if d else 0)
    return A


@pytest.fixture(scope="module")
def h():
    a = bsp.BspAtom(device=0)
    yield a
    a.close()


@pytest.fixture(scope="module")
def oracle_pencils():
    """the oracle's H_l and S (oracle/bsp_oracle.c: the reference's MATRIX_SVT restated), independent of the library"""
    from oracle import oracle as O

    b = O.make_basis(kind_grid=0, k=7, nfun=1000, rb=500.0)
    m = O.matrix_svt(b, lmax=max(LS), par=O.pot_params(0, 1.0))
    return {l: O.hamiltonian(m["T"], m["U"][:, :, l], m["V"]) for l in LS}, m["S"]


@pytest.fixture(scope="module")
def cfg2(h):
    a = host_basis(kind_grid=0, k=7, nfun=1000, rb=500.0)
    prob = bsp.Problem(k=a.k, nfun=a.nfun, nkp=a.nkp, ka=a.ka, rt=a.rt, pot_kind=bsp.POT_COULOMB, pot_par=(1.0,))
    band = h.MATRIX_SVT(prob)   # the device's own S, H0, Q (upper bands), and R
    mats = {}
    for l in LS:
        cl = float(l * (l + 1))
        H = dense_from_upper(band["H0"]) + cl * dense_from_upper(band["Q"])
        mats[l] = (H, cl)
    S = dense_from_upper(band["S"])
    return prob, band, S, mats


def upload(h, prob, nvec=1000):
    h.batch_upload([(prob, l) for l in LS], nvec=nvec)


def eigpairs(h, prob):
    upload(h, prob)
    h.batch_run()
    E, Cb, info = np.empty(4000), np.empty(4000 * 1000), np.zeros(4, np.int32)
    h.batch_download(E, Cb, info)
    assert np.all(info == 0)
    return [(E[i * 1000:(i + 1) * 1000], Cb[i * 10 ** 6:(i + 1) * 10 ** 6].reshape(1000, 1000, order="F")) for i in range(4)]


@pytest.mark.parametrize("kind", ["real", "complex"])
def test_cfg2_against_lapack_spectral_sum_and_replay(h, cfg2, emul, oracle_pencils, kind):
    prob, band, S, mats = cfg2
    Ho, So = oracle_pencils
    pairs = eigpairs(h, prob)
    rng = np.random.default_rng(7 if kind == "real" else 8)
    iprob, z, rhs = [], [], []
    for i, l in enumerate(LS):
        w = pairs[i][0]
        if kind == "real":
            zz = shifts_across(w, 6, rng)
        else:
            zz = w[0] + abs(w[0]) + rng.uniform(0.05, 2.0, 6) + 1j * np.array([1e-3, 1e-1] * 3)
        iprob += [i] * 6
        z += list(zz)
        rhs += list(rng.standard_normal((6, 1000)) * np.exp(-np.linspace(0.0, 25.0, 1000)))
    X, info, berr = h.shifted_solve(iprob, np.array(z), rhs)
    assert np.all(info == 0) and np.all(berr <= BERR_BAR), (info, berr)
    for s in range(len(z)):
        H, cl = mats[LS[iprob[s]]]
        ref_dev = lapack_solve(H, S, z[s], rhs[s], 6)
        assert rel_err(X[s], ref_dev) <= REL_LAPACK
        # against LAPACK on the oracle's pencil: the library's assembly agrees with the oracle's to ~1e-13 entrywise,
        # and the bar adds what that difference does to LAPACK's own solution (measured here, itself required small)
        ref_orc = lapack_solve(Ho[LS[iprob[s]]], So, z[s], rhs[s], 6)
        sens = rel_err(ref_dev, ref_orc)
        assert sens <= 1e-6
        assert rel_err(X[s], ref_orc) <= REL_LAPACK + 2.0 * sens
        w, Cv = pairs[iprob[s]]
        assert rel_err(X[s], Cv @ ((Cv.T @ rhs[s]) / (w - z[s]))) <= REL_SPECTRAL_DEVICE
    # bit for bit the CPU replay, on the device's own bands with H_l = fma(c_l, Q, H0) formed as the device forms it
    for i, l in enumerate(LS):
        sel = [s for s in range(len(z)) if iprob[s] == i][:3]
        Xr, ir, br, _ = replay(emul, dense_from_upper(band["H0"]), S, 6, np.array([z[s] for s in sel]),
                               np.array([rhs[s] for s in sel])[:, :, None], Q=dense_from_upper(band["Q"]), cl=mats[l][1])
        assert np.array_equal(ir, info[sel])
        assert np.array_equal(bits(br), bits(berr[sel]))
        for k, s in enumerate(sel):
            assert np.array_equal(bits(Xr[k, :, 0]), bits(X[s])), (l, s)


def test_hydrogen_polarisability(h, cfg2):
    prob, band, S, mats = cfg2
    pairs = eigpairs(h, prob)
    E0, C0 = pairs[0][0][0], pairs[0][1][:, 0]
    R = dense_from_upper(band["R"])
    b = R @ C0
    X, info, berr = h.shifted_solve([1], [E0], [b])
    assert info[0] == 0
    assert abs(2.0 / 3.0 * b @ X[0] - 4.5) < 1e-8
    # dynamic: alpha(w) = 1/3 b^T [x(E0 + w) + x(E0 - w)] = sum over states of the l = 1 pencil (bspatom_dipole)
    E1, C1 = pairs[1]
    kd = 6
    Rg = np.zeros((2 * kd + 1, 1000), order="F")
    for j in range(1000):
        for i in range(max(0, j - kd), min(1000, j + kd + 1)):
            Rg[kd + i - j, j] = R[i, j]
    d = h.dipole(Rg, C1, C0[:, None])[:, 0]
    for om in (0.05, 0.2, 0.3):
        X, info, _ = h.shifted_solve([1, 1], [E0 + om, E0 - om], [b, b])
        assert np.all(info == 0)
        alpha = (b @ X[0] + b @ X[1]) / 3.0
        sos = 2.0 / 3.0 * np.sum(d ** 2 * (E1 - E0) / ((E1 - E0) ** 2 - om ** 2))
        assert abs(alpha - sos) <= 1e-7 * abs(sos), (om, alpha, sos)


def band_pencils():
    rng = np.random.default_rng(20261022)
    out = [(*fem_hydrogen(2000, 1, 60.0), 1, 1, "U"), (*fem_hydrogen(4001, 1, 80.0), 1, 1, "L"), (*fem_hydrogen(2, 1, 10.0), 1, 1, "U")]
    for n, ka, kb, uplo in ((2, 1, 2, "U"), (6, 5, 2, "L"), (300, 9, 4, "U"), (500, 2, 7, "L"), (200, 0, 3, "U")):
        out.append((*random_pencil(rng, n, ka, kb), ka, kb, uplo))
    return out


def store(M, k, uplo):
    n = M.shape[0]
    ab = np.zeros((k + 1, n), order="F")
    for d in range(min(k, n - 1) + 1):
        if uplo == "U":
            ab[k - d, d:] = np.diagonal(M, d)
        else:
            ab[d, :n - d] = np.diagonal(M, d)
    return ab


def test_band_pencils_mixed_groups_any_order(h, emul):
    cases = band_pencils()
    h.band_upload([(store(A, ka, u), store(Bm, kb, u), u) for A, Bm, ka, kb, u in cases], nvec=0)
    rng = np.random.default_rng(3)
    iprob, z, rhs = [], [], []
    for i, (A, Bm, ka, kb, u) in enumerate(cases):
        w = eigh(A, Bm, eigvals_only=True)
        for zz in list(shifts_across(w, 3, rng, top=w[-1])) + [w[0] + 0.3 + 0.05j]:
            iprob.append(i)
            z.append(zz)
            rhs.append(rng.standard_normal(A.shape[0]))
    order = rng.permutation(len(z))
    iprob, z, rhs = [iprob[k] for k in order], np.array(z), [rhs[k] for k in order]
    z = z[order]
    X, info, berr = h.shifted_solve(iprob, z, rhs)
    assert np.all(info == 0) and np.all(berr <= BERR_BAR)
    for s in range(len(z)):
        A, Bm, ka, kb, _ = cases[iprob[s]]
        assert rel_err(X[s], lapack_solve(A, Bm, z[s], rhs[s], max(ka, kb))) <= REL_LAPACK
    # real systems alone, through the real entry, against the replay bit for bit
    for s in [k for k in range(len(z)) if z[k].imag == 0][:6]:
        A, Bm, ka, kb, _ = cases[iprob[s]]
        Xs, i1, b1 = h.shifted_solve([iprob[s]], [z[s].real], [rhs[s]])
        Xr, ir, br, _ = replay(emul, A, Bm, band_width(ka, kb, A.shape[0]), [z[s].real], rhs[s][None, :, None])
        assert np.array_equal(bits(Xs[0]), bits(Xr[0, :, 0])) and i1[0] == ir[0]


@pytest.mark.parametrize("nrhs", [0, 1, 3, 9])
def test_right_hand_side_counts(h, cfg2, nrhs):
    prob, band, S, mats = cfg2
    upload(h, prob, nvec=0)
    rng = np.random.default_rng(nrhs)
    z = [-0.3, 0.01, 0.77]
    rhs = [rng.standard_normal((1000, nrhs)) for _ in z]
    X, info, berr = h.shifted_solve([2, 2, 2], z, rhs)
    assert np.all(info == 0)
    for s in range(3):
        for c in range(nrhs):
            assert rel_err(X[s][:, c], lapack_solve(mats[17][0], S, z[s], rhs[s][:, c], 6)) <= REL_LAPACK
            Xc, *_ = h.shifted_solve([2], [z[s]], [rhs[s][:, c]])
            assert np.array_equal(bits(Xc[0]), bits(X[s][:, c]))


def test_many_shifts_chunking_and_independence(h, cfg2):
    """1000 shifts on one pencil; a mixed call in arbitrary order; every system's bits are those of the same system
    solved alone and under another chunking (option shifted_chunk)"""
    prob, band, S, mats = cfg2
    upload(h, prob, nvec=0)
    rng = np.random.default_rng(11)
    z1 = np.linspace(-0.6, 3.0, 1000) + 1.234e-5
    b1 = [rng.standard_normal(1000) for _ in z1]
    X1, i1, e1 = h.shifted_solve([0] * 1000, z1, b1)
    assert np.all((i1 == 0) | (i1 == 1001))
    assert np.mean(i1 == 0) > 0.99
    # the solutions themselves: every shift at least 1e-4 (relative) from the spectrum, against LAPACK
    H0 = mats[0][0]
    w0 = eigh(H0, S, eigvals_only=True)
    far = [s for s in range(1000) if np.min(np.abs(w0 - z1[s])) > 1e-4 * max(abs(z1[s]), 1e-2)]
    assert len(far) > 500
    for s in far[::10]:
        assert i1[s] == 0 and e1[s] <= BERR_BAR
        assert rel_err(X1[s], lapack_solve(H0, S, z1[s], b1[s], 6)) <= REL_LAPACK
    iprob = rng.integers(0, 4, 700)
    z = rng.uniform(-0.5, 2.0, 700) + 1j * rng.choice([1e-3, 1e-1], 700)
    rhs = [rng.standard_normal(1000) + 1j * rng.standard_normal(1000) for _ in z]
    Xa, ia, ba = h.shifted_solve(iprob, z, rhs)
    try:
        h.set_option("shifted_chunk", 128)
        Xb, ib, bb = h.shifted_solve(iprob, z, rhs)
    finally:
        h.set_option("shifted_chunk", 0)
    assert np.array_equal(ia, ib) and np.array_equal(bits(ba), bits(bb))
    for s in range(700):
        assert np.array_equal(bits(Xa[s]), bits(Xb[s]))
    for s in (0, 17, 699):
        Xs, is_, bs = h.shifted_solve([iprob[s]], [z[s]], [rhs[s]])
        assert np.array_equal(bits(Xs[0]), bits(Xa[s])) and bs[0] == ba[s]


def test_hard_cases(h, cfg2):
    A, Bm = np.array([[0.0, 1.0], [1.0, 0.0]]), np.eye(2)
    Bind = np.diag([1.0, -1.0, 1.0])
    h.band_upload([(store(A, 1, "U"), store(Bm, 0, "U"), "U"), (store(np.eye(3), 0, "U"), store(Bind, 0, "U"), "U")], nvec=0)
    X, info, berr = h.shifted_solve([0, 0, 1], [0.0, 0.5, 0.1], [np.ones(2), np.ones(2), np.ones(3)])
    assert info[0] == 1 and np.all(np.isnan(X[0]))
    assert info[1] == 0 and np.allclose(X[1], np.linalg.solve(A - 0.5 * Bm, np.ones(2)), rtol=1e-14)
    assert info[2] == 3 + 2 and np.all(np.isnan(X[2]))      # the upload dropped it: B indefinite at pivot 2
    prob, band, S, mats = cfg2
    w = eigpairs(h, prob)[0][0]
    X, info, berr = h.shifted_solve([0, 0, 0], w[[0, 5, 400]], [np.ones(1000)] * 3)
    for s in range(3):
        if 1 <= info[s] <= 1000:
            continue
        assert (info[s] == 1001) == (berr[s] > BERR_BAR)
        assert np.all(np.isfinite(X[s]))


def raw(h, nsys, iprob, z, nrhs, B, X, info, berr=None, cplx=False):
    f = h.lib.bspatom_shifted_solve_z if cplx else h.lib.bspatom_shifted_solve
    p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None   # noqa: E731
    return f(h._h, nsys, p(iprob), p(z), nrhs, p(B), p(X), p(info), p(berr))


def test_errors_and_state(cfg2):
    prob, band, S, mats = cfg2
    g = bsp.BspAtom(device=0)
    try:
        ip, z, B, X, info = np.zeros(1, np.int32), np.zeros(1), np.ones(1000), np.zeros(1000), np.zeros(1, np.int32)
        assert raw(g, 1, ip, z, 1, B, X, info) == _lib.ESTATE
        g.batch_upload([(prob, l) for l in LS], nvec=1000)
        assert raw(g, -1, ip, z, 1, B, X, info) == -2
        assert raw(g, 1, None, z, 1, B, X, info) == -3
        assert raw(g, 1, np.array([4], np.int32), z, 1, B, X, info) == -3
        assert raw(g, 1, np.array([-1], np.int32), z, 1, B, X, info) == -3
        assert raw(g, 1, ip, None, 1, B, X, info) == -4
        assert raw(g, 1, ip, np.array([np.nan]), 1, B, X, info) == -4
        assert raw(g, 1, ip, np.array([0.0, np.inf]), 1, np.ones(2000), np.zeros(2000), info, cplx=True) == -4
        assert raw(g, 1, ip, z, -1, B, X, info) == -5
        assert raw(g, 1, ip, z, 1, None, X, info) == -6
        assert raw(g, 1, ip, z, 1, B, None, info) == -7
        assert raw(g, 1, ip, z, 1, B, X, None) == -8
        assert np.all(X == 0)
        # a shifted solve before batch_run leaves that run's bits alone, and one after it the resident results
        g.shifted_solve([0, 3], [-0.2, 0.4], [np.ones(1000), np.ones(1000)])
        g.batch_run()
        E1, C1, I1 = np.empty(4000), np.empty(4 * 10 ** 6), np.zeros(4, np.int32)
        g.batch_download(E1, C1, I1)
        v1 = g.batch_verify()
        A_band = np.asfortranarray(np.vstack([np.zeros((6, 1000)), band["R"]]))
        D1 = g.dipole_chain_resident(A_band[:13], 0, 4, 20)
        g.shifted_solve([1, 2], [0.1 + 0.01j, -0.4], [np.ones(1000), np.ones(1000)])
        E2, C2, I2 = np.empty(4000), np.empty(4 * 10 ** 6), np.zeros(4, np.int32)
        g.batch_download(E2, C2, I2)
        assert np.array_equal(bits(E1), bits(E2)) and np.array_equal(bits(C1), bits(C2)) and np.array_equal(I1, I2)
        assert g.batch_verify() == v1
        assert np.array_equal(bits(g.dipole_chain_resident(A_band[:13], 0, 4, 20)), bits(D1))
        ref = bsp.BspAtom(device=0)
        try:
            ref.batch_upload([(prob, l) for l in LS], nvec=1000)
            ref.batch_run()
            E3, C3, I3 = np.empty(4000), np.empty(4 * 10 ** 6), np.zeros(4, np.int32)
            ref.batch_download(E3, C3, I3)
        finally:
            ref.close()
        assert np.array_equal(bits(E1), bits(E3)) and np.array_equal(bits(C1), bits(C3)) and np.array_equal(I1, I3)
        st = g.stats()
        assert st["ms_shifted_solve"] > 0 and 1 <= st["shifted_refinement_steps"] <= 5
    finally:
        g.close()


def test_sizes_follow_every_call_that_replaces_the_batch(h, cfg2):
    """the operand shapes come from the library's resident batch, whichever call put it there"""
    prob, band, S, mats = cfg2
    a = host_basis(kind_grid=0, k=7, nfun=500, rb=250.0)
    small = bsp.Problem(k=a.k, nfun=a.nfun, nkp=a.nkp, ka=a.ka, rt=a.rt, pot_kind=bsp.POT_COULOMB, pot_par=(1.0,))
    h.batch_upload([(small, 0)], nvec=0)
    assert list(h.batch_sizes()) == [a.nfun]
    h.solve_batch([(prob, l) for l in LS], nvec=1)          # upload + run of 1000-row pencils
    assert list(h.batch_sizes()) == [1000] * 4
    with pytest.raises(ValueError):
        h.shifted_solve([0], [0.1], [np.ones(a.nfun)])
    rhs = np.random.default_rng(1).standard_normal(1000)
    X, info, berr = h.shifted_solve([1], [0.1], [rhs])
    assert info[0] == 0 and rel_err(X[0], lapack_solve(mats[1][0], S, 0.1, rhs, 6)) <= REL_LAPACK
    A, Bm = random_pencil(np.random.default_rng(2), 40, 3, 2)
    h.solve_band_batch([(store(A, 3, "U"), store(Bm, 2, "U"), "U")], nvec=1)
    assert list(h.batch_sizes()) == [40]
    X, info, berr = h.shifted_solve([0], [-7.0], [np.ones(40)])
    assert info[0] == 0 and rel_err(X[0], np.linalg.solve(A + 7.0 * Bm, np.ones(40))) <= REL_LAPACK
    g = bsp.BspAtom(device=0)
    try:
        g.adopt(bsp.BspInputs.from_values(kind_grid=2, k=7, nfun=100, rb=500.0, rmax=60.0, lmax=2))
        g.SOLVE_SYSTEM()
        n = g.nfun
        assert list(g.batch_sizes()) == [n] * 3
        X, info, berr = g.shifted_solve([1], [g.Enl[0, 0]], [np.ones(n)])
        assert info[0] == 0 and berr[0] <= BERR_BAR
    finally:
        g.close()


def test_device_operands_and_unwritten_systems(h):
    """B and X in device memory give the host path's bits; a system with a failed pivot leaves its X alone"""
    import torch

    A, Bm = random_pencil(np.random.default_rng(5), 300, 4, 2)
    Z2 = np.array([[0.0, 1.0], [1.0, 0.0]])
    h.band_upload([(store(A, 4, "L"), store(Bm, 2, "L"), "L"), (store(Z2, 1, "U"), store(np.eye(2), 0, "U"), "U")], nvec=0)
    rng = np.random.default_rng(6)
    iprob = [0, 1, 0, 1]
    z = np.array([-3.0 + 0.2j, 0.0, 0.37 - 0.01j, 0.5 + 0.0j])
    rhs = [rng.standard_normal(300) + 1j * rng.standard_normal(300), np.ones(2, complex),
           rng.standard_normal(300) + 0j, np.ones(2, complex)]
    Xh, ih, bh = h.shifted_solve(iprob, z, rhs)
    assert list(ih) == [0, 1, 0, 0]
    Bd = torch.tensor(np.concatenate(rhs), dtype=torch.complex128, device="cuda")
    Xd = torch.full((604,), 7.0 + 7.0j, dtype=torch.complex128, device="cuda")
    idv, bdv = h.shifted_solve_ptrs(iprob, z, 1, Bd.data_ptr(), Xd.data_ptr(), complex_=True)
    torch.cuda.synchronize()
    x = Xd.cpu().numpy()
    assert np.array_equal(idv, ih) and np.array_equal(bits(bdv), bits(bh))
    assert np.array_equal(bits(x[:300]), bits(Xh[0])) and np.all(x[300:302] == 7.0 + 7.0j)
    assert np.array_equal(bits(x[302:602]), bits(Xh[2])) and np.array_equal(bits(x[602:]), bits(Xh[3]))


def test_more_systems_than_one_layout_grid_holds(h):
    """2.2 million systems of order 3: more slots than 65535 tiles of 32, so the call must be chunked"""
    A, Bm = random_pencil(np.random.default_rng(9), 3, 1, 1)
    h.band_upload([(store(A, 1, "U"), store(Bm, 1, "U"), "U")], nvec=0)
    nsys = 2_200_000
    rng = np.random.default_rng(10)
    z = rng.uniform(-6.0, -4.0, nsys)          # below the spectrum: well conditioned
    B = rng.standard_normal(3 * nsys)
    X = np.full_like(B, np.nan)
    info, berr = h.shifted_solve_ptrs(np.zeros(nsys, np.int32), z, 1, B.ctypes.data, X.ctypes.data)
    assert np.all(info == 0) and np.all(berr <= BERR_BAR)
    for s in list(range(0, nsys, 99_991)) + [nsys - 1]:
        ref = np.linalg.solve(A - z[s] * Bm, B[3 * s:3 * s + 3])
        assert rel_err(X[3 * s:3 * s + 3], ref) <= 1e-13
