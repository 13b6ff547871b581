"""ctypes binding of libbspatom.so (include/bspatom.h).  No torch types cross this boundary.

There is no CPU fallback: if the library is missing, or no CUDA device is present, loading /
handle creation raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BSPATOM_LIB") or os.path.join(_HERE, "libbspatom.so")  # override: A/B builds only

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)

ENODEVICE, ECUDA, EUNSUPPORTED, ESTATE, ENOMEM = 1001, 1002, 1003, 1004, 1005

EXPORTS = [
    "bspatom_create", "bspatom_destroy", "bspatom_last_error", "bspatom_version", "bspatom_set_option",
    "bspatom_alloc_host", "bspatom_free_host",
    "bspatom_assemble_band", "bspatom_solve_batch", "bspatom_batch_upload", "bspatom_batch_run",
    "bspatom_batch_download", "bspatom_get_selection", "bspatom_batch_verify", "bspatom_dsygv_", "bspatom_dipole", "bspatom_dipole_chain", "bspatom_dipole_chain_resident",
    "bspatom_create_multi", "bspatom_destroy_multi", "bspatom_last_error_multi", "bspatom_set_option_multi", "bspatom_solve_batch_multi",
    "bspatom_trans_amp_hermitian", "bspatom_assemble_zaij", "bspatom_wavefunction", "bspatom_wavefunction_resident", "bspatom_get_stats",
    "bspatom_band_upload", "bspatom_solve_band_batch", "bspatom_dsbgv_",
]


class BspProblem(C.Structure):
    """struct bsp_problem of include/bspatom.h"""

    _fields_ = [
        ("k", C.c_int), ("nfun", C.c_int), ("nkp", C.c_int), ("ka", C.c_int),
        ("rt", _dp), ("xg", _dp), ("wg", _dp),
        ("pot_kind", C.c_int), ("pot_par", C.c_double * 8),
        ("v_tab", _dp),
        ("l", C.c_int), ("ul_extra", C.c_double), ("nvec", C.c_int),
        ("sel_mode", C.c_int), ("sel_extra", C.c_int), ("sel_group", C.c_int),
        ("sel_ecut_a", C.c_double), ("sel_ecut_b", C.c_double),
    ]


class BspBandPencil(C.Structure):
    """struct bsp_band_pencil of include/bspatom.h"""

    _fields_ = [
        ("n", C.c_int), ("ka", C.c_int), ("kb", C.c_int), ("uplo", C.c_char),
        ("AB", _dp), ("ldab", C.c_int), ("BB", _dp), ("ldbb", C.c_int), ("nvec", C.c_int),
    ]


class BspAtomError(RuntimeError):
    pass


_lib = None


def load():
    """Load the CUDA library; raises if it has not been built (run __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BspAtomError(f"{LIB_PATH} is missing: build it with `python -m bspatom_b200.build` "
                           "(there is no CPU fallback for this path)")
    L = C.CDLL(LIB_PATH)
    H = C.c_void_p
    L.bspatom_create.argtypes = [C.POINTER(H), C.c_int]
    L.bspatom_destroy.argtypes = [H]
    L.bspatom_last_error.argtypes = [H]
    L.bspatom_last_error.restype = C.c_char_p
    L.bspatom_version.restype = C.c_int
    L.bspatom_set_option.argtypes = [H, C.c_char_p, C.c_double]
    L.bspatom_alloc_host.argtypes = [C.c_size_t]
    L.bspatom_alloc_host.restype = C.c_void_p
    L.bspatom_free_host.argtypes = [C.c_void_p]
    L.bspatom_free_host.restype = None
    L.bspatom_assemble_band.argtypes = [H, C.POINTER(BspProblem)] + [C.c_void_p] * 8
    L.bspatom_solve_batch.argtypes = [H, C.c_int, C.POINTER(BspProblem), C.c_void_p, C.c_void_p, C.c_void_p]
    L.bspatom_batch_upload.argtypes = [H, C.c_int, C.POINTER(BspProblem)]
    L.bspatom_batch_run.argtypes = [H]
    L.bspatom_batch_download.argtypes = [H, C.c_void_p, C.c_void_p, C.c_void_p]
    L.bspatom_batch_verify.argtypes = [H, _dp]
    L.bspatom_get_selection.argtypes = [H, C.c_void_p]
    L.bspatom_dsygv_.argtypes = [_ip, C.c_char_p, C.c_char_p, _ip, C.c_void_p, _ip, C.c_void_p, _ip,
                                 C.c_void_p, C.c_void_p, _ip, _ip]
    L.bspatom_dsygv_.restype = None
    L.bspatom_dipole.argtypes = [H, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                 C.c_void_p]
    L.bspatom_dipole_chain.argtypes = [H, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.bspatom_trans_amp_hermitian.argtypes = [H, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                              C.c_void_p]
    L.bspatom_create_multi.argtypes = [C.POINTER(C.c_void_p), C.c_int, _ip]
    L.bspatom_destroy_multi.argtypes = [C.c_void_p]
    L.bspatom_last_error_multi.argtypes = [C.c_void_p]
    L.bspatom_last_error_multi.restype = C.c_char_p
    L.bspatom_set_option_multi.argtypes = [C.c_void_p, C.c_char_p, C.c_double]
    L.bspatom_solve_batch_multi.argtypes = [C.c_void_p, C.c_int, C.POINTER(BspProblem), C.c_void_p, C.c_void_p, _ip]
    L.bspatom_assemble_zaij.argtypes = [H, C.POINTER(BspProblem), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    L.bspatom_wavefunction.argtypes = [H, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_double,
                                       C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.bspatom_dipole_chain_resident.argtypes = [H, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.bspatom_wavefunction_resident.argtypes = [H, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int,
                                                C.c_void_p, C.c_void_p]
    L.bspatom_get_stats.argtypes = [H, _dp, C.c_int]
    L.bspatom_band_upload.argtypes = [H, C.c_int, C.POINTER(BspBandPencil)]
    L.bspatom_solve_band_batch.argtypes = [H, C.c_int, C.POINTER(BspBandPencil), C.c_void_p, C.c_void_p, C.c_void_p]
    L.bspatom_dsbgv_.argtypes = [C.c_char_p, C.c_char_p, _ip, _ip, _ip, C.c_void_p, _ip, C.c_void_p, _ip, C.c_void_p,
                                 C.c_void_p, _ip, C.c_void_p, _ip]
    L.bspatom_dsbgv_.restype = None
    _lib = L
    return L


def check(lib, handle, rc, what):
    if rc == 0:
        return
    msg = lib.bspatom_last_error(handle).decode() if handle else ""
    names = {ENODEVICE: "no CUDA device (this path has no CPU fallback)", ECUDA: "CUDA error",
             EUNSUPPORTED: "B-spline order k outside the compiled range 3..10", ESTATE: "call order",
             ENOMEM: "out of device memory"}
    raise BspAtomError(f"{what} failed: rc={rc} {names.get(rc, 'invalid argument' if rc < 0 else '')} {msg}")
