"""GPU: the banded product and the FP64 DMMA GEMM (csrc/bsp_gemm.cuh) against exact references, through the public
entries dipole, dipole_chain, trans_amp_hermitian and batch_verify.

Exact cases use integer-valued operands (entries in [-8, 8], integer bands): every product and every partial sum is an
integer below 2^53, so the result is exact whatever the summation order and must match the integer product bit for bit.
That pins every GEMM tile variant (gemm_variant 1..4 and the automatic pick), ragged M / N edges, the K tail of every
size mod 16 and both the 16-byte (even leading dimensions and strides) and the 8-byte copy path."""
import numpy as np
import pytest

import bspatom_b200 as bsp
from cases import EPS, band_to_dense_sym, host_basis

pytestmark = pytest.mark.gpu

RNG = np.random.default_rng(20261020)


def ints(*shape):
    return RNG.integers(-8, 9, size=shape)


def exact_tn(a, b):
    """a^T b of integer arrays, exactly, as float64.  int64 matmul for small products; numpy's float64 product for big
    ones (as exact: every partial sum is an integer below 2^53, checked here, so no summation order can round)."""
    bound = a.shape[0] * float(np.abs(a).max(initial=0)) * float(np.abs(b).max(initial=0))
    assert bound < 2.0 ** 53
    if a.shape[0] * a.shape[1] * b.shape[1] <= 2e7:
        return (a.T.astype(np.int64) @ b.astype(np.int64)).astype(np.float64)
    return a.T.astype(np.float64) @ b.astype(np.float64)


def general_band(A, kd):
    """dense (n, n) -> LAPACK general band (2kd+1, n), AB[kd+i-j, j] = A[i, j]"""
    n = A.shape[0]
    ab = np.zeros((2 * kd + 1, n), order="F")
    for d in range(-kd, kd + 1):           # A[j+d, j] lives in row kd+d
        j = np.arange(max(0, -d), min(n, n - d))
        ab[kd + d, j] = A[j + d, j]
    return ab


def int_band(n, kd):
    return np.triu(np.tril(ints(n, n), kd), -kd)


@pytest.fixture
def variant(atom):
    """gemm_variant is process-wide: every test that forces one puts the automatic pick back"""
    try:
        yield lambda v: atom.set_option("gemm_variant", v)
    finally:
        atom.set_option("gemm_variant", 0)


# (M, N, K): M, N in {1, 7, 8, 15, 16, 17, 63, 64, 65, 127, 128, 129, 1000}, K in {1, 3, 8, 15, 16, 17, 33, 1000, 1001}
GEMM_SHAPES = [(1, 1, 1), (7, 8, 3), (8, 7, 8), (15, 16, 15), (16, 15, 16), (17, 17, 17), (63, 64, 33), (64, 65, 1000),
               (65, 63, 1001), (127, 128, 17), (128, 129, 16), (129, 127, 33), (1, 1000, 1001), (1000, 1, 8),
               (1000, 129, 1000), (129, 1000, 1001), (1000, 1000, 1000)]


@pytest.mark.parametrize("v", [0, 1, 2, 3, 4])
def test_dgemm_exact_every_variant(atom, variant, v):
    """kd = 0 identity band: dipole is the bare GEMM Cf^T Ci"""
    variant(v)
    for M, N, K in GEMM_SHAPES:
        Cf, Ci = ints(K, M), ints(K, N)
        D = atom.dipole(np.ones((1, K)), Cf.astype(np.float64), Ci.astype(np.float64))
        assert np.array_equal(D, exact_tn(Cf, Ci)), (v, M, N, K)


@pytest.mark.parametrize("v", [0, 1, 2, 3, 4])
def test_dgemm_exact_k_tail_of_every_size(atom, variant, v):
    """K = 16 .. 33: the last k-tile holds 0 .. 15 valid columns; even K takes the 16-byte copies, odd K the 8-byte ones"""
    variant(v)
    for K in range(16, 34):
        Cf, Ci = ints(K, 17), ints(K, 9)
        D = atom.dipole(np.ones((1, K)), Cf.astype(np.float64), Ci.astype(np.float64))
        assert np.array_equal(D, exact_tn(Cf, Ci)), (v, K)


@pytest.mark.parametrize("nl", [3, 8, 50])
@pytest.mark.parametrize("nvec", [1000, 999, 130])
def test_dipole_chain_exact_batched(atom, nl, nvec):
    """batched GEMM of the cfg5 chain at n = 1000, automatic pick (variant 2 for 8 and 50 blocks of 1000 or 999 vectors,
    variant 3 for the others): the block strides n * nvec are even (1000, 130) and odd (999)"""
    n, kd = 1000, 6
    A = int_band(n, kd)
    Cs = [ints(n, nvec) for _ in range(nl)]
    D = atom.dipole_chain(general_band(A, kd).astype(np.float64), [c.astype(np.float64) for c in Cs])
    assert D.shape == (nl - 1, nvec, nvec)
    for l in range(nl - 1):
        Y = A.astype(np.int64) @ Cs[l]            # banded: cheap in int64
        assert np.array_equal(D[l], exact_tn(Cs[l + 1], Y)), l


@pytest.mark.parametrize("n,nf,ni", [(203, 65, 63), (1000, 999, 130)])
def test_trans_amp_hermitian_exact(atom, n, nf, ni):
    """complex path: Gaussian-integer upper band; ZHEMV('U') semantics (lower triangle from the upper one, imaginary part of
    the diagonal ignored) restated on the integer parts: T = Cf^T Re(A_h) Ci + i Cf^T Im(A_h) Ci"""
    kd = 6
    re, im = np.triu(np.tril(ints(n, n), kd)), np.triu(np.tril(ints(n, n), kd))
    zab = np.zeros((kd + 1, n), dtype=np.complex128, order="F")
    for d in range(kd + 1):                    # A[j-d, j] lives in row kd-d
        j = np.arange(d, n)
        zab[kd - d, j] = re[j - d, j] + 1j * im[j - d, j]
    Ar = re + np.triu(re, 1).T
    Ai = np.triu(im, 1) - np.triu(im, 1).T
    Cf, Ci = ints(n, nf), ints(n, ni)
    T = atom.trans_amp_hermitian(zab, Cf.astype(np.float64), Ci.astype(np.float64))
    ref = exact_tn(Cf, Ar.astype(np.int64) @ Ci) + 1j * exact_tn(Cf, Ai.astype(np.int64) @ Ci)
    assert np.array_equal(T, ref)


@pytest.mark.parametrize("kd", [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 14, 81])
def test_band_times_dense_exact(atom, kd):
    """Y = A Ci for every templated half bandwidth (2..9), the generic kernel (0, 1, 10 and up; 14 is the first that needs
    more than 48 KB of shared memory, 81 the last below 200 KB); Cf = I so that D = Y"""
    nvs = [1, 15, 16, 17, 33]
    for i, n in enumerate(x for x in (1, 2, 127, 128, 129, 1000) if x > kd):
        nv = nvs[(i + kd) % len(nvs)]
        A, Ci = int_band(n, kd), ints(n, nv)
        D = atom.dipole(general_band(A, kd), np.eye(n), Ci.astype(np.float64))
        assert np.array_equal(D, (A.astype(np.int64) @ Ci).astype(np.float64)), (kd, n, nv)


def test_band_too_wide_is_an_error_not_a_crash(atom):
    n, kd = 1000, 82
    with pytest.raises(bsp.BspAtomError):
        atom.dipole(general_band(int_band(n, kd), kd), np.eye(n)[:, :3], ints(n, 5).astype(np.float64))
    Ci = ints(n, 5)                            # the handle keeps working
    D = atom.dipole(np.ones((1, n)), np.eye(n), Ci.astype(np.float64))
    assert np.array_equal(D, Ci.astype(np.float64))


@pytest.fixture(scope="module")
def cfg5_vectors(atom, oracle):
    """GPU eigenvectors of the N = 1000 cfg2 pencils, l = 0, 1, 49, 50, and the oracle's dipole operator R"""
    a = host_basis(kind_grid=0, k=7, nfun=1000, rb=500.0)
    Es, Cs, info = atom.solve_batch([(a.problem(), l) for l in (0, 1, 49, 50)])
    assert not info.any()
    b = oracle.make_basis(kind_grid=0, k=7, nfun=1000, rb=500.0)
    R = oracle.matrix_svt(b, lmax=0, want_u=False)["R"]
    return {l: np.asarray(c) for l, c in zip((0, 1, 49, 50), Cs)}, R


@pytest.mark.parametrize("l0", [0, 49])
def test_cfg5_shape_against_extended_precision(atom, variant, cfg5_vectors, l0):
    """D = C_{l0+1}^T R C_{l0} of the N = 1000 spectra, automatic pick and every forced variant, against the product in
    np.longdouble: bar 1e-12 |row| |col| (the cfg5 bar)"""
    Cv, R = cfg5_vectors
    Ci, Cf = Cv[l0], Cv[l0 + 1]
    n, kd = R.shape[0], 6
    Rl, Cil = R.astype(np.longdouble), Ci.astype(np.longdouble)
    Y = np.zeros_like(Cil)
    for d in range(-kd, kd + 1):               # banded R Ci in extended precision
        i = np.arange(max(0, -d), min(n, n - d))
        Y[i] += Rl[i, i + d][:, None] * Cil[i + d]
    ref = Cf.astype(np.longdouble).T @ Y
    scale = np.linalg.norm(Cf, axis=0)[:, None] * np.linalg.norm(R @ Ci, axis=0)[None, :]
    Rb = general_band(R, kd)
    for v in (0, 1, 2, 3, 4):
        variant(v)
        D = atom.dipole(Rb, Cf, Ci)
        err = float(np.max(np.abs((D - ref).astype(np.float64)) / scale))
        assert err < 1e-12, (v, err)


# ---------------------------------------------------------------------------------------------------------------------
# bspatom_batch_verify against the same quantities computed on the host
# ---------------------------------------------------------------------------------------------------------------------
def upload(atom, items, nvecs=None, select=None):
    """batch_upload with one nvec per item (the wrapper takes one nvec per batch)"""
    from bspatom_b200.host import build_problem_array
    from bspatom_b200._lib import check

    if nvecs is None:
        atom.batch_upload(items, select=select)
        return
    arr, keep = build_problem_array(items, None, select)
    arr.rec["nvec"] = nvecs
    check(atom.lib, atom._h, atom.lib.bspatom_batch_upload(atom._h, len(items), arr), "bspatom_batch_upload")
    atom._last_items = items


def run_and_download(atom, items, nvecs):
    atom.batch_run()
    nf = np.array([p.nfun for p, _ in items])
    E, Cb, info = np.empty(nf.sum()), np.full(int((nf * nvecs).sum()), np.nan), np.zeros(len(items), np.int32)
    atom.batch_download(E, Cb, info)
    assert not info.any()
    eo, co = np.concatenate(([0], np.cumsum(nf))), np.concatenate(([0], np.cumsum(nf * nvecs)))
    return ([E[eo[i]:eo[i + 1]] for i in range(len(items))],
            [Cb[co[i]:co[i + 1]].reshape((nf[i], nvecs[i]), order="F") for i in range(len(items))])


def host_verify(atom, items, Es, Cs, nv):
    """max scaled residual, max |C^T S C - I| (np.longdouble, on the library's own bands) and their rounding allowances:
    64 eps times the norms the device sums (|H| |c| + |E| |S| |c| per residual, |C|^T |S| |C| per Gram entry)"""
    res = orth = res_tol = orth_tol = 0.0
    bands = {}
    for (p, l), E, Cm, k in zip(items, Es, Cs, nv):
        if id(p) not in bands:
            m = atom.MATRIX_SVT(p)
            bands[id(p)] = tuple(band_to_dense_sym(m[x], p.nfun) for x in ("S", "H0", "Q"))
        S, H0, Q = bands[id(p)]
        H = H0 + (l * (l + 1)) * Q
        c, e = Cm[:, :k], E[:k]
        cl, Hl, Sl, el = c.astype(np.longdouble), H.astype(np.longdouble), S.astype(np.longdouble), e.astype(np.longdouble)
        SC = Sl @ cl
        r = np.abs(Hl @ cl - SC * el).max(axis=0) / np.maximum(1, np.abs(el))
        res = max(res, float(r.max()))
        orth = max(orth, float(np.abs(cl.T @ SC - np.eye(k)).max()))
        w = (np.abs(H) @ np.abs(c) + np.abs(e) * (np.abs(S) @ np.abs(c))).max(axis=0) / np.maximum(1, np.abs(e))
        res_tol = max(res_tol, 64 * EPS * float(w.max()))
        orth_tol = max(orth_tol, 64 * EPS * float((np.abs(c).T @ (np.abs(S) @ np.abs(c))).max()))
    return res, orth, res_tol, orth_tol


def assert_verify_agrees(atom, items, Es, Cs, nv):
    v = atom.batch_verify()
    res, orth, res_tol, orth_tol = host_verify(atom, items, Es, Cs, nv)
    assert v["eigenpairs_checked"] == int(np.sum(nv))
    assert abs(v["max_scaled_residual"] - res) <= res_tol, (v, res, res_tol)
    assert abs(v["max_orthonormality_defect"] - orth) <= orth_tol, (v, orth, orth_tol)
    assert v["not_ascending"] == 0.0
    return v, orth


def test_batch_verify_agrees_with_the_host(atom):
    a = host_basis(kind_grid=0, k=7, nfun=300, rb=150.0)
    p = a.problem()
    items = [(p, l) for l in range(6)]
    nv = np.full(6, 300)
    upload(atom, items)
    Es, Cs = run_and_download(atom, items, nv)
    assert_verify_agrees(atom, items, Es, Cs, nv)
    # the fast schedule leaves |C^T S C - I| ~ 1e-8, far above rounding: the device must see the same defect
    atom.set_option("vec_tol", 1e300)
    try:
        upload(atom, items)
        Es, Cs = run_and_download(atom, items, nv)
    finally:
        atom.set_option("vec_tol", 1e-12)
    v, orth = assert_verify_agrees(atom, items, Es, Cs, nv)
    assert orth > 1e-10
    assert abs(v["max_orthonormality_defect"] - orth) <= 1e-3 * orth


def test_batch_verify_mixed_shapes_nvec_and_selection(atom):
    """two groups (N = 300, k = 7 and N = 200, k = 5) with per-pencil nvec: the Gram GEMM runs over pencils of equal nvec
    only; then a device-side selection: only the selected columns exist and are counted"""
    a1 = host_basis(kind_grid=0, k=7, nfun=300, rb=150.0)
    a2 = host_basis(kind_grid=1, k=5, nfun=200, rb=100.0)
    p1, p2 = a1.problem(), a2.problem()
    items = [(p1, 0), (p1, 1), (p2, 0), (p1, 2), (p1, 3), (p2, 1), (p1, 4), (p2, 2)]
    nv = np.array([300, 300, 200, 120, 120, 37, 300, 37])
    upload(atom, items, nv)
    Es, Cs = run_and_download(atom, items, nv)
    assert_verify_agrees(atom, items, Es, Cs, nv)

    items = [(p1, l) for l in range(6)]
    full = np.full(6, 300)
    upload(atom, items, select=bsp.Selection.from_kind_pi(0.5, 3))
    Es, Cs = run_and_download(atom, items, full)
    nsel = atom.selection()
    assert 0 < nsel.min() and nsel.max() < 300
    assert_verify_agrees(atom, items, Es, Cs, nsel)
