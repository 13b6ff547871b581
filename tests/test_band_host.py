"""No GPU: the host side of the band-pencil entry points.  struct bsp_band_pencil as the C compiler lays it out against
its ctypes mirror, the argument checks and leading dimensions of bspatom_b200.host.band_pencil_array, the LAPACK -i
codes of bspatom_dsbgv_ (all decided before a device is needed), and no CPU fallback."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import bspatom_b200 as bsp
from bspatom_b200 import _lib
from bspatom_b200.host import band_pencil_array

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _has_gpu():
    import torch

    return torch.cuda.is_available()


def test_band_pencil_layout_matches_header(tmp_path):
    fields = [f for f, _ in _lib.BspBandPencil._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "bspatom.h"\nint main(void){\n'
                   'printf("%zu\\n", sizeof(bsp_band_pencil));\n' +
                   "".join('printf("%%zu\\n", offsetof(bsp_band_pencil, %s));\n' % f for f in fields) + "return 0;}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    out = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert out[0] == ctypes.sizeof(_lib.BspBandPencil)
    for f, off in zip(fields, out[1:]):
        assert getattr(_lib.BspBandPencil, f).offset == off, f


def test_band_pencil_array_fields_and_leading_dimensions():
    n = 12
    AB = np.asfortranarray(np.arange(4.0 * n).reshape(4, n))
    buf = np.zeros((6, n), order="F")
    BB = buf[:2]                                   # Fortran view into a taller buffer: ldbb = 6, no copy
    Cview = np.ascontiguousarray(AB)               # C order: copied into Fortran order
    arr, keep, ns, nvs = band_pencil_array([(AB, BB), (Cview, BB, "L")], nvec=5)
    p0, p1 = arr[0], arr[1]
    assert (p0.n, p0.ka, p0.kb, p0.uplo, p0.ldab, p0.ldbb, p0.nvec) == (n, 3, 1, b"U", 4, 6, 5)
    assert (p1.uplo, p1.ldab) == (b"L", 4)
    assert ctypes.addressof(p0.AB.contents) == AB.ctypes.data
    assert ctypes.addressof(p0.BB.contents) == BB.ctypes.data
    assert ctypes.addressof(p1.AB.contents) != Cview.ctypes.data
    assert np.array_equal(keep[2], Cview) and keep[2].flags.f_contiguous
    assert ns == [n, n] and nvs == [5, 5]
    # a scalar nvec is capped at n, per-pencil values are passed as given (the library checks the range)
    assert band_pencil_array([(AB, BB)], nvec=100)[3] == [n]
    assert band_pencil_array([(AB, BB)], nvec=[100])[3] == [100]
    assert band_pencil_array([(AB, BB)])[3] == [n]


def test_band_pencil_array_keeps_its_copies_alive():
    """operands that are not Fortran-ordered float64 are copied; the struct array must keep those copies alive (a
    ctypes pointer stored in a struct does not), or it points into freed memory once the caller drops the list"""
    import gc

    rng = np.random.default_rng(1)
    AB, BB = rng.uniform(size=(3, 200)), rng.uniform(size=(2, 200))       # C order: copied
    arr = band_pencil_array([(AB, BB), (AB.astype(np.float32), BB[:, ::-1])])[0]   # float32, negative stride: copied
    gc.collect()
    junk = [np.full(AB.shape, 123.0) for _ in range(256)]
    p0 = arr[0]
    got = np.ctypeslib.as_array(p0.AB, shape=(200 * 3,)).reshape((3, 200), order="F")
    assert np.array_equal(got, AB)
    got = np.ctypeslib.as_array(p0.BB, shape=(200 * 2,)).reshape((2, 200), order="F")
    assert np.array_equal(got, BB)
    got = np.ctypeslib.as_array(arr[1].AB, shape=(200 * 3,)).reshape((3, 200), order="F")
    assert np.array_equal(got, AB.astype(np.float32).astype(np.float64))
    got = np.ctypeslib.as_array(arr[1].BB, shape=(200 * 2,)).reshape((2, 200), order="F")
    assert np.array_equal(got, BB[:, ::-1])
    del junk


@pytest.mark.parametrize("bad, match", [
    (lambda AB, BB: [(AB[0], BB)], "2-D"),
    (lambda AB, BB: [(AB, BB[:, :-1])], "columns"),
    (lambda AB, BB: [(AB, BB, "UP")], "uplo"),
    (lambda AB, BB: [(AB,)], "expected"),
])
def test_band_pencil_array_rejects_malformed_input(bad, match):
    AB, BB = np.zeros((3, 8), order="F"), np.ones((2, 8), order="F")
    with pytest.raises(ValueError, match=match):
        band_pencil_array(bad(AB, BB))
    with pytest.raises(ValueError, match="entries"):
        band_pencil_array([(AB, BB)], nvec=[1, 2])


def test_dsbgv_lapack_argument_codes():
    """argument checks in DSBGV's order; none of them needs a device"""
    lib = _lib.load()
    n = 6
    AB, BB = np.zeros((3, n), order="F"), np.ones((2, n), order="F")
    w, Z, work = np.zeros(n), np.zeros((n, n), order="F"), np.zeros(3 * n)
    ci = lambda v: ctypes.byref(ctypes.c_int(v))  # noqa: E731
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731

    def call(jobz=b"V", uplo=b"U", nn=n, ka=2, kb=1, ab=AB, ldab=3, bb=BB, ldbb=2, ldz=n, ww=w):
        info = ctypes.c_int(99)
        lib.bspatom_dsbgv_(jobz, uplo, ci(nn), ci(ka), ci(kb), vp(ab) if ab is not None else None, ci(ldab),
                           vp(bb) if bb is not None else None, ci(ldbb), vp(ww) if ww is not None else None, vp(Z), ci(ldz),
                           vp(work), ctypes.byref(info))
        return info.value

    assert call(jobz=b"X") == -1
    assert call(uplo=b"X") == -2
    assert call(nn=-1) == -3
    assert call(ka=-1) == -4 and call(ka=10) == -4
    assert call(kb=3) == -5 and call(kb=-1) == -5
    assert call(ab=None) == -6
    assert call(ldab=2) == -7
    assert call(bb=None) == -8
    assert call(ldbb=1) == -9
    assert call(ww=None) == -10
    assert call(ldz=n - 1) == -12 and call(jobz=b"N", ldz=0) == -12
    assert call(nn=0) == 0                                      # quick return
    nan = AB.copy(order="F")
    nan[2, 3] = np.nan                                          # stored diagonal of A
    assert call(ab=nan) == -6
    nan = BB.copy(order="F")
    nan[0, 4] = np.inf                                          # stored superdiagonal of B
    assert call(bb=nan) == -8
    w2, Z2, info = bsp.dsbgv(BB, AB)                            # kb > ka from the shapes
    assert info == -5


def test_band_entries_have_no_cpu_fallback(tmp_path):
    if _has_gpu():
        pytest.skip("a device is present")
    n = 6
    AB, BB = np.ones((1, n), order="F"), np.ones((1, n), order="F")
    w, Z, info = bsp.dsbgv(AB, BB)
    assert info < -100
    w, Z, info = bsp.dsbgv(AB, BB, jobz="N")
    assert info < -100 and Z is None
    with pytest.raises(bsp.BspAtomError, match="no CUDA device"):
        bsp.BspAtom(device=0)
    exe = str(tmp_path / "c_band_driver")
    libdir = os.path.join(ROOT, "bspatom_b200")
    subprocess.check_call(["gcc", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe,
                           os.path.join(ROOT, "tests", "c_band_driver.c"), "-L", libdir, "-lbspatom",
                           "-Wl,-rpath," + libdir, "-lm"])
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 77 and "no CUDA device" in r.stdout
    P = _lib.BspBandPencil
    want = "sizeof(bsp_band_pencil) = %d, offsets ka %d kb %d uplo %d AB %d ldab %d BB %d ldbb %d nvec %d" % (
        ctypes.sizeof(P), P.ka.offset, P.kb.offset, P.uplo.offset, P.AB.offset, P.ldab.offset, P.BB.offset,
        P.ldbb.offset, P.nvec.offset)
    assert want in r.stdout, r.stdout
