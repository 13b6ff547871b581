"""Host side of the B200 path, mirroring the reference driver's interface.

The reference is a Fortran program whose hot path is two argument-less subroutines that talk
through module globals (``CALL MATRIX_SVT`` Bsp_Atom.f90:72, ``CALL SOLVE_SYSTEM`` Bsp_Atom.f90:75).
No Fortran compiler exists in this image, so -- as the task prescribes for a compiled reference
whose toolchain is absent -- the host above the C-ABI is written here, keeping the reference's
names and meaning: ``BspAtom`` holds what MOD_GRID / MOD_BSPLINES / MOD_PHOTOION hold
(Modules.f90:21-58,207-236) and offers READ_INPUTS, GRID, MATRIX_SVT, SOLVE_SYSTEM, WRITE_WF,
TRANS_AMP.  The Fortran binding a maintainer would add instead is in INTEGRATION.md.

Everything numeric below the knot vector runs on the GPU through libbspatom.so; this module only
parses input, builds knots (GRID stays on the host in the reference too) and moves buffers.
"""
from __future__ import annotations

import ctypes as C
import math
import re
from dataclasses import dataclass, field
from typing import Iterable, List, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import BspAtomError, BspBandPencil, BspProblem

POT_COULOMB, POT_ROGERS, POT_SIMONS_FUES, POT_YUKAWA, POT_TIETZ, POT_TABLE = 0, 1, 2, 10, 11, -1

# Simons-Fues Bl(0:3) for Rb, ReadInputs.f90:136-139
_BL_RB = (0.72657, 0.47095, -0.55508, -0.04008)


# --------------------------------------------------------------------------------------
# input: three namelists on stdin (ReadInputs.f90:15-21)
# --------------------------------------------------------------------------------------
_NML_DEFAULTS = {
    "VARS_BSP": dict(KIND_GRID=0, ra=0.0, rb=0.0, rmax=0.0, k=0, ka=0, nfun=0, KIND_BC1=0, KIND_BC2=0, nfib=1),
    "VARS_TISE": dict(KIND_POT=0, n0_ini=1, l_ini=0, m_ini=0, l_fin=0, lmax=0, Emax_fin=-1.0, Zatom=1.0,
                      KIND_EGR=0, KIND_NLM=0),
    "VARS_FIELD": dict(KIND_PI=0),
}


def _fortran_value(tok: str):
    t = tok.strip().rstrip(",")
    if re.fullmatch(r"[+-]?\d+", t):
        return int(t)
    return float(t.replace("D", "E").replace("d", "e"))


def parse_namelists(text: str) -> dict:
    """Parse the bsp_0.inp format: '!' comment lines, ``&GROUP name=value ... &end`` blocks."""
    lines = [ln for ln in text.splitlines() if not ln.lstrip().startswith("!")]
    body = " ".join(lines)
    out = {g: dict(d) for g, d in _NML_DEFAULTS.items()}
    for m in re.finditer(r"&(\w+)(.*?)(?:&end|/)", body, flags=re.S | re.I):
        group = m.group(1).upper()
        vals = out.setdefault(group, {})
        known = {k.lower(): k for k in vals}
        for kv in re.finditer(r"(\w+)\s*=\s*([^\s,=]+)", m.group(2)):
            name = known.get(kv.group(1).lower(), kv.group(1))
            vals[name] = _fortran_value(kv.group(2))
    return out


def _nint(x: float) -> int:
    """Fortran NINT: round half away from zero."""
    return int(math.floor(x + 0.5)) if x >= 0 else -int(math.floor(-x + 0.5))


@dataclass
class Problem:
    """One radial problem instance: knots + potential (what MATRIX_SVT reads from the modules)."""

    k: int
    nfun: int
    nkp: int
    ka: int
    rt: np.ndarray
    xg: Optional[np.ndarray] = None
    wg: Optional[np.ndarray] = None
    pot_kind: int = POT_COULOMB
    pot_par: Sequence[float] = (1.0,)
    v_tab: Optional[np.ndarray] = None
    bl: Optional[Sequence[float]] = None  # Bl(0:lmax) for KIND_POT=2


class BspInputs:
    """What READ_INPUTS + GRID leave in MOD_GRID / MOD_BSPLINES / MOD_PHOTOION: pure host logic,
    no GPU needed (the reference keeps these on the host as well)."""

    def __init__(self):
        self.KIND_GRID = 0
        self.KIND_BC1 = self.KIND_BC2 = 0
        self.KIND_POT = 0
        self.KIND_PI = 0
        self.ra = self.rb = self.rmax = 0.0
        self.k = self.ka = self.nfun = self.nkp = self.nointv = 0
        self.nbc1 = self.nbc2 = self.nintv_exp = self.nintv_lin = 0
        self.lmax = self.l_ini = self.l_fin = 0
        self.n0_ini = 1
        self.Zatom = 1.0
        self.Emax_fin = -1.0
        self.pot_par = np.zeros(8)
        self.Bl = None
        self.rt = None

    @classmethod
    def from_values(cls, kind_grid=0, k=7, ka=0, nfun=100, ra=0.0, rb=500.0, rmax=0.0, kind_bc1=0, kind_bc2=0,
                    zatom=1.0, kind_pot=0, lmax=0):
        a = cls()
        a.KIND_GRID, a.k, a.ka, a.nfun = kind_grid, k, ka, nfun
        a.KIND_BC1, a.KIND_BC2 = kind_bc1, kind_bc2
        a.ra, a.rb, a.rmax = ra, rb, rmax
        a.Zatom, a.KIND_POT, a.lmax = zatom, kind_pot, lmax
        a.set_sizes()
        a.set_potential()
        a.GRID()
        return a

    # ---- READ_INPUTS (ReadInputs.f90:1-145) ---------------------------------------------
    def READ_INPUTS(self, text: str):
        nml = parse_namelists(text)
        b, t, f = nml["VARS_BSP"], nml["VARS_TISE"], nml["VARS_FIELD"]
        self.KIND_GRID, self.ra, self.rb, self.rmax = int(b["KIND_GRID"]), float(b["ra"]), float(b["rb"]), float(b["rmax"])
        self.k, self.ka, self.nfun = int(b["k"]), int(b["ka"]), int(b["nfun"])
        self.KIND_BC1, self.KIND_BC2 = int(b["KIND_BC1"]), int(b["KIND_BC2"])
        self.set_sizes()
        self.KIND_POT = int(t["KIND_POT"])
        self.n0_ini, self.l_ini, self.l_fin = int(t["n0_ini"]), int(t["l_ini"]), int(t["l_fin"])
        self.lmax = int(t["lmax"])
        self.Emax_fin, self.Zatom = float(t["Emax_fin"]), float(t["Zatom"])
        if self.l_fin > self.lmax:                       # ReadInputs.f90:87
            self.lmax = self.l_fin
        self.KIND_PI = int(f.get("KIND_PI", 0))
        self.set_potential()
        return self

    def set_sizes(self):
        """derived sizes, ReadInputs.f90:39-69"""
        k = self.k
        if self.ka == 0:
            self.ka = k + 3
        self.nbc1 = k if self.KIND_BC1 != 0 else k - 1
        self.nbc2 = k if self.KIND_BC2 != 0 else k - 1
        self.nkp = self.nfun + k
        self.nointv = self.nkp - self.nbc1 - self.nbc2 + 1
        self.gsize = self.rb - self.ra
        if self.KIND_GRID == 2:
            dx = self.gsize / self.nointv
            imax = _nint((self.rmax - self.ra) / dx)
            self.nintv_exp = 3 * imax
            self.nintv_lin = self.nointv - imax
            self.nointv = self.nintv_exp + self.nintv_lin
            self.nkp = self.nointv + self.nbc1 + self.nbc2 - 1
            self.nfun = self.nkp - k

    def set_potential(self):
        """potential tables, ReadInputs.f90:95-141"""
        par = np.zeros(8)
        par[0] = self.Zatom
        self.Bl = None
        if self.KIND_POT == POT_ROGERS:
            numn = (2, 8, 8)
            aj = ((0.8855, 0.2549, -0.0901, 0.0), (0.3386, 1.1323, -0.4904, 0.0), (0.1437, 0.9129, -0.6940, 0.2503))
            ntot = 0
            for i in range(3):
                ntot += numn[i]
                xn = float(self.Zatom - ntot)
                if xn == 0.0:
                    xn = 1.0
                suman = 0.0
                for j in range(4):
                    suman = suman + aj[i][j] / (xn ** j)
                par[5 + i] = (xn + 1.0) * suman
                par[2 + i] = numn[i]
            par[1] = ntot
        elif self.KIND_POT == POT_SIMONS_FUES:
            bl = np.zeros(max(self.lmax, 3) + 1)
            bl[:4] = _BL_RB
            self.Bl = bl
        self.pot_par = par

    # ---- GRID (grid.f90:1-63): knots stay a host computation ---------------------------
    def GRID(self):
        nkp, nbc1, nbc2, ra, rb = self.nkp, self.nbc1, self.nbc2, self.ra, self.rb
        rt = np.zeros(nkp)
        rt[:nbc1] = ra
        rt[nkp - nbc2:] = rb
        if self.KIND_GRID == 0:
            for i in range(nbc1 + 1, nkp - nbc2 + 1):
                rt[i - 1] = ra + float(i - nbc1) * self.gsize / float(self.nointv)
        elif self.KIND_GRID == 1:
            delta = 0.01
            hin = math.log(self.gsize / delta) / float(self.nointv - 1)
            rt[nbc1] = delta
            j = 1
            for i in range(nbc1 + 2, nkp - nbc2 + 1):
                rt[i - 1] = rt[nbc1] * math.exp(hin * j)
                j += 1
        elif self.KIND_GRID == 2:
            delta = 0.01
            hin = math.log((self.rmax - ra) / delta) / float(self.nintv_exp - 1)
            rt[nbc1] = delta
            j = 1
            for i in range(2, self.nintv_exp + 1):
                rt[i + nbc1 - 1] = delta * math.exp(hin * j)
                j += 1
            dr = (rb - self.rmax) / float(self.nintv_lin)
            for i in range(self.nintv_exp + 1, self.nointv + 1):
                rt[i + nbc1 - 1] = self.rmax + float(i - self.nintv_exp) * dr
        else:
            raise ValueError("KIND_GRID must be 0, 1 or 2")
        self.rt = rt
        return rt

    def problem(self) -> Problem:
        if self.rt is None:
            self.GRID()
        return Problem(k=self.k, nfun=self.nfun, nkp=self.nkp, ka=self.ka, rt=self.rt, pot_kind=self.KIND_POT,
                       pot_par=tuple(self.pot_par), bl=self.Bl)


class BspAtom(BspInputs):
    """State + entry points of the reference driver for the hot path (PROGRAM BSP_ATOM_PI)."""

    def __init__(self, device: int = 0):
        super().__init__()
        self.lib = _lib.load()
        self._h = C.c_void_p()
        rc = self.lib.bspatom_create(C.byref(self._h), int(device))
        _lib.check(self.lib, None, rc, "bspatom_create")
        self.device = device
        self.Enl = None   # (nfun, lmax+1)  eigenvalues per l   (Enl, matrices.f90:294)
        self.cinl = None  # list over l of (nfun, nvec) eigenvector blocks (cinl, matrices.f90:369)
        self.info = None

    def adopt(self, inp: "BspInputs"):
        """take over sizes / knots / potential from a BspInputs"""
        for k_, v in vars(inp).items():
            setattr(self, k_, v)
        return self

    # ---- lifetime ---------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self.lib.bspatom_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name: str, value: float):
        _lib.check(self.lib, self._h, self.lib.bspatom_set_option(self._h, name.encode(), float(value)),
                   "bspatom_set_option")

    def stats(self) -> dict:
        out = (C.c_double * 24)()
        self.lib.bspatom_get_stats(self._h, out, 24)
        keys = ["launches", "rounds", "iters", "ms_assembly", "ms_eigenvalues", "ms_eigenvectors", "ms_finalize",
                "ms_total", "ms_k_round", "ms_k_factor", "ms_k_back", "ms_k_assembly",
                "n_k_round", "n_k_factor", "n_k_back", "n_k_assembly", "wall_ms_upload", "wall_ms_run",
                "wall_ms_download", "chunks_redone", "selected_third_solve", "wall_ms_copy_tail", "c_bytes_copied",
                "ms_resident_contraction"]
        return dict(zip(keys, list(out)))

    # ---- MATRIX_SVT (matrices.f90:1-200) ------------------------------------------------
    def MATRIX_SVT(self, prob: Optional[Problem] = None) -> dict:
        """Banded S, H0=T+V, Q, T, V, R, Rinv (upper band, (k, nfun) Fortran order) and D
        (general band (2k-1, nfun)).  Uij(:,:,l) = [l(l+1)+2Bl(l)] Q."""
        prob = prob or self.problem()
        keep: list = []
        cp = _to_c_problem(prob, 0, 0, keep)
        k, n = prob.k, prob.nfun
        names = ["S", "H0", "Q", "T", "V", "R", "Rinv"]
        out = {nm: np.zeros((k, n), order="F") for nm in names}
        out["D"] = np.zeros((2 * k - 1, n), order="F")
        ptrs = [out[nm].ctypes.data_as(C.c_void_p) for nm in names + ["D"]]
        rc = self.lib.bspatom_assemble_band(self._h, C.byref(cp), *ptrs)
        _lib.check(self.lib, self._h, rc, "bspatom_assemble_band")
        self.band = out
        return out

    # ---- SOLVE_SYSTEM core (matrices.f90:242-265) --------------------------------------
    def SOLVE_SYSTEM(self, nvec: Optional[int] = None, device_select: Optional[bool] = None):
        """Loop l = 0..lmax of the reference, as ONE batched call.  Fills Enl, cinl, info.
        Raises like the reference STOPs (matrices.f90:250-254) when info != 0.
        device_select (default: on for KIND_PI >= 3 with a given Emax_fin): the reference keeps ctemp(:, 1:ntemp, l)
        only (matrices.f90:296-334); the same rule then runs on the device right after the eigenvalue stage, and only
        those columns are refined and copied (cinl blocks keep the shape (nfun, nvec); columns >= ntemp(l) are unset)."""
        prob = self.problem()
        ls = list(range(self.lmax + 1))
        if device_select is None:
            device_select = self.KIND_PI >= 3 and self.Emax_fin != -1.0
        select = Selection.from_kind_pi(self.Emax_fin, self.KIND_PI) if device_select else None
        E, Cs, info = self.solve_batch([(prob, l) for l in ls], nvec=nvec, select=select)
        self.info = info
        bad = [(l, i) for l, i in zip(ls, info) if i != 0]
        if bad:
            raise BspAtomError("ERROR DIAGONALIZING THE MATRIX! info=%d  l = %d" % (bad[0][1], bad[0][0]))
        self.Enl = np.stack(E, axis=1)
        self.cinl = Cs
        # bookkeeping of matrices.f90:269-346 on the gathered eigenpairs (host side, like the reference)
        self.sel = None
        if self.KIND_PI != 0:
            from . import postproc

            self.sel = postproc.select_states(self.Enl, self.KIND_PI, self.l_ini, self.l_fin, self.Emax_fin)
            self.Emax_fin = self.sel.Emax_fin
        return self.Enl, self.cinl

    def write_outputs(self, directory: str = "."):
        """Enl.dat (matrices.f90:239-265) and, for KIND_PI >= 3, Eigenvec_All.dat (matrices.f90:366-378)."""
        import os

        from . import postproc

        postproc.write_enl(os.path.join(directory, "Enl.dat"), self.Enl)
        if self.KIND_PI >= 3 and self.sel is not None:
            cinl = postproc.collect_cinl(self.cinl, self.sel)
            postproc.write_eigenvec_all(os.path.join(directory, "Eigenvec_All.dat"), cinl)

    def solve_batch(self, items: Iterable, nvec: Optional[int] = None, want_vectors: bool = True,
                    out_E: Optional[np.ndarray] = None, out_C: Optional[np.ndarray] = None,
                    select: Optional["Selection"] = None):
        """items: iterable of (Problem, l).  Returns (list of E arrays, list of C arrays, info).
        select: device-side state selection (Selection): C blocks keep the shape (nfun, nvec) but only the first
        ``self.selection()[i]`` columns of block i are computed and copied out."""
        items = list(items)
        arr, keep = build_problem_array(items, nvec, select)
        nfs, nvs = arr.rec["nfun"].astype(np.int64), arr.rec["nvec"].astype(np.int64)
        n_e = int(nfs.sum())
        n_c = int((nfs * nvs).sum())
        self._last_items = items
        E = out_E if out_E is not None else pinned_empty(n_e)
        Cbuf = (out_C if out_C is not None else pinned_empty(n_c)) if want_vectors else None
        info = np.zeros(len(items), dtype=np.int32)
        rc = self.lib.bspatom_solve_batch(self._h, len(items), arr, E.ctypes.data_as(C.c_void_p),
                                          Cbuf.ctypes.data_as(C.c_void_p) if Cbuf is not None else None,
                                          info.ctypes.data_as(C.c_void_p))
        _lib.check(self.lib, self._h, rc, "bspatom_solve_batch")
        eo = np.concatenate(([0], np.cumsum(nfs)))
        co = np.concatenate(([0], np.cumsum(nfs * nvs)))
        Es = [E[eo[i]:eo[i + 1]] for i in range(len(items))]
        Cs = []
        if Cbuf is not None:
            Cs = [Cbuf[co[i]:co[i + 1]].reshape((int(nfs[i]), int(nvs[i])), order="F") for i in range(len(items))]
        return Es, Cs, info

    # staged variant: keeps the batch resident in HBM (bench.py times batch_run alone)
    def selection(self) -> np.ndarray:
        """eigenvectors computed per problem by the last run (bspatom_get_selection)"""
        n = len(self._last_items)
        out = np.zeros(n, dtype=np.int32)
        _lib.check(self.lib, self._h, self.lib.bspatom_get_selection(self._h, out.ctypes.data_as(C.c_void_p)),
                   "bspatom_get_selection")
        return out

    def batch_upload(self, items: Iterable, nvec: Optional[int] = None, select: Optional["Selection"] = None):
        items = list(items)
        self._last_items = items
        arr, keep = build_problem_array(items, nvec, select)
        rc = self.lib.bspatom_batch_upload(self._h, len(items), arr)
        _lib.check(self.lib, self._h, rc, "bspatom_batch_upload")
        self._resident = (items, arr.rec["nvec"].copy())

    def batch_run(self):
        _lib.check(self.lib, self._h, self.lib.bspatom_batch_run(self._h), "bspatom_batch_run")

    # ---- caller-supplied band pencils (DSBGV semantics) ---------------------------------
    def band_upload(self, pencils: Iterable, nvec=None, uplo: str = "U"):
        """bspatom_band_upload: pencils are (AB, BB) or (AB, BB, uplo) with AB (ka+1, n) and BB (kb+1, n) in LAPACK
        band storage (see band_pencil_array).  batch_run / batch_download / batch_verify / selection /
        dipole_chain_resident then apply as after batch_upload."""
        arr, keep, ns, _ = band_pencil_array(pencils, nvec, uplo)   # keep: the arrays arr points into
        rc = self.lib.bspatom_band_upload(self._h, len(ns), arr)
        _lib.check(self.lib, self._h, rc, "bspatom_band_upload")
        self._last_items = ns

    def solve_band_batch(self, pencils: Iterable, nvec=None, want_vectors: bool = True, uplo: str = "U",
                         out_E: Optional[np.ndarray] = None, out_C: Optional[np.ndarray] = None):
        """bspatom_solve_band_batch: A x = E B x for every (AB, BB[, uplo]) pencil.  Returns (list of E arrays, list of
        (n, nvec) C blocks, info) like solve_batch; a pencil with info > n (B not positive definite) keeps whatever
        its E / C slots held.  Pinned out_E / out_C (pinned_empty) are filled chunk by chunk."""
        arr, keep, ns, nvs = band_pencil_array(pencils, nvec, uplo)   # keep: the arrays arr points into
        nfs, nvs = np.asarray(ns, dtype=np.int64), np.asarray(nvs, dtype=np.int64)
        self._last_items = ns
        E = out_E if out_E is not None else pinned_empty(int(nfs.sum()))
        Cbuf = (out_C if out_C is not None else pinned_empty(int((nfs * nvs).sum()))) if want_vectors else None
        info = np.zeros(len(ns), dtype=np.int32)
        rc = self.lib.bspatom_solve_band_batch(self._h, len(ns), arr, E.ctypes.data_as(C.c_void_p),
                                               Cbuf.ctypes.data_as(C.c_void_p) if Cbuf is not None else None,
                                               info.ctypes.data_as(C.c_void_p))
        _lib.check(self.lib, self._h, rc, "bspatom_solve_band_batch")
        eo = np.concatenate(([0], np.cumsum(nfs)))
        co = np.concatenate(([0], np.cumsum(nfs * nvs)))
        Es = [E[eo[i]:eo[i + 1]] for i in range(len(ns))]
        Cs = []
        if Cbuf is not None:
            Cs = [Cbuf[co[i]:co[i + 1]].reshape((int(nfs[i]), int(nvs[i])), order="F") for i in range(len(ns))]
        return Es, Cs, info

    def batch_download(self, E: np.ndarray, Cbuf: Optional[np.ndarray], info: np.ndarray):
        rc = self.lib.bspatom_batch_download(self._h, E.ctypes.data_as(C.c_void_p),
                                             Cbuf.ctypes.data_as(C.c_void_p) if Cbuf is not None else None,
                                             info.ctypes.data_as(C.c_void_p))
        _lib.check(self.lib, self._h, rc, "bspatom_batch_download")

    def batch_verify(self) -> dict:
        """Device-side check of the resident batch: max scaled residual over every eigenpair, max |C^T S C - I|
        over every pencil, ascending spectra (bspatom_batch_verify)."""
        out = (C.c_double * 4)()
        _lib.check(self.lib, self._h, self.lib.bspatom_batch_verify(self._h, out), "bspatom_batch_verify")
        return {"max_scaled_residual": out[0], "max_orthonormality_defect": out[1], "not_ascending": out[2],
                "eigenpairs_checked": int(out[3])}

    def batch_download_ptrs(self, E_ptr: int, C_ptr: Optional[int], info: Optional[np.ndarray] = None):
        """bspatom_batch_download with raw (host or DEVICE) destination addresses, e.g. torch CUDA tensors'
        data_ptr(): the eigenpairs stay on the GPU (send buffers of the NCCL gather)."""
        rc = self.lib.bspatom_batch_download(self._h, C.c_void_p(E_ptr) if E_ptr else None,
                                             C.c_void_p(C_ptr) if C_ptr else None,
                                             info.ctypes.data_as(C.c_void_p) if info is not None else None)
        _lib.check(self.lib, self._h, rc, "bspatom_batch_download")

    # ---- WRITE_WF (Bsp_Atom.f90:101-152) ------------------------------------------------
    def WRITE_WF(self, ci: np.ndarray, npts: int = 10000):
        ci = np.asarray(ci, dtype=np.float64)
        if ci.ndim == 1:
            ci = ci[:, None]
        ci = np.asfortranarray(ci)
        if ci.shape[0] != self.nfun:
            raise ValueError("ci must have nfun rows")
        nvec = ci.shape[1]
        r = np.empty(npts + 1)
        psi = np.empty((npts + 1, nvec), order="F")
        rt = np.ascontiguousarray(self.rt)
        rc = self.lib.bspatom_wavefunction(self._h, self.k, self.nfun, self.nkp, rt.ctypes.data_as(C.c_void_p),
                                           self.ra, self.rb, npts, nvec, ci.ctypes.data_as(C.c_void_p),
                                           r.ctypes.data_as(C.c_void_p), psi.ctypes.data_as(C.c_void_p))
        _lib.check(self.lib, self._h, rc, "bspatom_wavefunction")
        return r, psi

    # ---- WRITEWF (WriteWF.f90:1-68): many wavefunctions of one l on the r-grid -----------------------
    def WRITEWF(self, n0: int, n1: int, l0: int, npts: int = 10000, literal: bool = True, path: Optional[str] = None):
        """The states WRITEWF writes to WFs.dat: n = 1 first, then n = n0 .. n1 (1-based) of cinl(:, :, l0), one column
        each, evaluated on r = ra + i (rb - ra)/npts in ONE launch of the wavefunction kernel.
        literal = True keeps the reference's coefficient indexing j = left - nbc1 + jfun (WriteWF.f90:38,51), which is
        one function higher than WRITE_WF's j = left - k + jfun when nbc1 = k - 1 (SURVEY.md 8(f) row f-1): the same
        kernel on the coefficient vectors shifted by k - nbc1; literal = False follows WRITE_WF.
        path: also write the file, FORMAT(100G20.10) (records longer than 100 items wrap like Fortran's format reversion)."""
        if self.cinl is None:
            raise BspAtomError("WRITEWF before SOLVE_SYSTEM")
        Cl = np.asarray(self.cinl[l0])
        cols = [0] + list(range(n0 - 1, n1))
        if max(cols) >= Cl.shape[1] or n0 < 1:
            raise ValueError("WRITEWF: states %d..%d outside the %d eigenvectors kept for l = %d" % (n0, n1, Cl.shape[1], l0))
        Csel = np.zeros((self.nfun, len(cols)), order="F")
        shift = (self.k - self.nbc1) if literal else 0
        Csel[: self.nfun - shift, :] = Cl[shift:, cols]
        r, fr = self.WRITE_WF(Csel, npts=npts)
        if shift == 1:
            # in the first knot interval the literal mapping also reaches j = 1 where WRITE_WF's j = 0 is skipped: it pairs
            # c(1) with bsp(1), the B-spline that READ_INPUTS dropped for the boundary condition, ((t1 - r)/(t1 - ra))^(k-1)
            t1 = float(self.rt[self.nbc1])
            first = r < t1
            fr[first, :] += np.outer(((t1 - r[first]) / (t1 - self.ra)) ** (self.k - 1), Cl[0, cols])
        elif shift > 1:
            raise BspAtomError("WRITEWF(literal=True): nbc1 = %d < k - 1 is not a configuration READ_INPUTS produces" % self.nbc1)
        if path is not None:
            from . import postproc

            with open(path, "w") as f:
                for i in range(npts + 1):
                    vals = [r[i]] + [fr[i, j] for j in range(fr.shape[1])]
                    for a in range(0, len(vals), 100):
                        f.write("".join(postproc.fortran_g(v, 20, 10) for v in vals[a:a + 100]) + "\n")
        return r, fr

    # ---- TRANS_AMP contraction (PhotoIon.f90:90-105) ------------------------------------
    def dipole(self, A_band: np.ndarray, Cf: np.ndarray, Ci: np.ndarray) -> np.ndarray:
        """D = Cf^T A Ci with A in general band storage (2kd+1, n)."""
        A_band = np.asfortranarray(A_band, dtype=np.float64)
        Cf = np.asfortranarray(Cf, dtype=np.float64)
        Ci = np.asfortranarray(Ci, dtype=np.float64)
        n = Cf.shape[0]
        kd = (A_band.shape[0] - 1) // 2
        D = np.empty((Cf.shape[1], Ci.shape[1]), order="F")
        rc = self.lib.bspatom_dipole(self._h, n, kd, A_band.ctypes.data_as(C.c_void_p), Cf.shape[1],
                                     Cf.ctypes.data_as(C.c_void_p), Ci.shape[1], Ci.ctypes.data_as(C.c_void_p),
                                     D.ctypes.data_as(C.c_void_p))
        _lib.check(self.lib, self._h, rc, "bspatom_dipole")
        return D


def _trans_amp_hermitian(self, zA_upper: np.ndarray, Cf: np.ndarray, Ci: np.ndarray) -> np.ndarray:
    """General (structured-light) branch of TRANS_AMP, PhotoIon.f90:218-232, for one angular block and all (bra, ket)
    pairs at once: T = Cf^T ZHEMV_U(zA) Ci (complex nf x ni), ZHEMV('U') semantics of ZHVMV (Modules.f90:398-425).
    zA_upper: complex upper band (kd+1, n), AB[kd+i-j, j] = zA[i, j]."""
    zA_upper = np.asfortranarray(zA_upper, dtype=np.complex128)
    Cf = np.asfortranarray(Cf, dtype=np.float64)
    Ci = np.asfortranarray(Ci, dtype=np.float64)
    n = Cf.shape[0]
    kd = zA_upper.shape[0] - 1
    T = np.empty((Cf.shape[1], Ci.shape[1]), dtype=np.complex128, order="F")
    rc = self.lib.bspatom_trans_amp_hermitian(self._h, n, kd, zA_upper.ctypes.data_as(C.c_void_p), Cf.shape[1],
                                              Cf.ctypes.data_as(C.c_void_p), Ci.shape[1],
                                              Ci.ctypes.data_as(C.c_void_p), T.ctypes.data_as(C.c_void_p))
    _lib.check(self.lib, self._h, rc, "bspatom_trans_amp_hermitian")
    return T


BspAtom.trans_amp_hermitian = _trans_amp_hermitian


def _matrix_svt_z(self, kind_pi: int, zIth: np.ndarray, ncomp_out: Optional[int] = None, prob: Optional[Problem] = None) -> np.ndarray:
    """KIND_PI >= 3 branch of MATRIX_SVT (matrices.f90:110-139, 164-175): the complex band matrices zAij from the
    angular integrals zIth(nkp, ka, nlm, nm, ncomp) the host tabulated (ZINT_TH, Ang_Ints.f90:544-600).
    Returns the general band (2k-1, nfun, nlm, nm, ncomp_out), AB[k-1+i-j, j] = zAij[i, j] (0-based), Fortran order."""
    prob = prob or self.problem()
    zIth = np.asfortranarray(zIth, dtype=np.complex128)
    if zIth.ndim != 5:
        raise BspAtomError("zIth must have the shape (nkp, ka, nlm, nm, ncomp)")
    nkp, ka, nlm, nm, ncomp = zIth.shape
    keep: list = []
    cp = _to_c_problem(prob, 0, 0, keep)
    if nkp != cp.nkp or ka != cp.ka:
        raise BspAtomError("zIth is tabulated on (nkp, ka) = (%d, %d), the problem has (%d, %d)" % (nkp, ka, cp.nkp, cp.ka))
    if ncomp_out is None:
        ncomp_out = min(4, ncomp) if kind_pi >= 5 else (4 if kind_pi == 4 else 2)
    zA = np.zeros((2 * prob.k - 1, prob.nfun, nlm, nm, ncomp_out), dtype=np.complex128, order="F")
    rc = self.lib.bspatom_assemble_zaij(self._h, C.byref(cp), int(kind_pi), nlm * nm, ncomp, zIth.ctypes.data_as(C.c_void_p),
                                        int(ncomp_out), zA.ctypes.data_as(C.c_void_p))
    _lib.check(self.lib, self._h, rc, "bspatom_assemble_zaij")
    return zA


BspAtom.MATRIX_SVT_Z = _matrix_svt_z


def _tormat_rvec(self, cinl: np.ndarray, R_upper: np.ndarray) -> np.ndarray:
    """TORMAT's matrix elements of r (TorusFuns.f90:127-158): rvecij(ni, li, nj, lj) = cinl(:,ni,li)^T Xij cinl(:,nj,lj)
    for ALL pairs in one band x dense product and one DMMA GEMM (the reference: (n1_max (lmax+1))^2 DSYMV + DDOT).
    cinl: (nfun, n1_max, lmax+1); R_upper: upper band (k, nfun) of Xij = int B_i r B_j (MATRIX_SVT()["R"]); like
    DSVMV('U') only the upper triangle of Xij is read."""
    cinl = np.asfortranarray(cinl, dtype=np.float64)
    n, n1, nl = cinl.shape
    kd = R_upper.shape[0] - 1
    A = np.zeros((2 * kd + 1, n), order="F")
    A[: kd + 1, :] = R_upper                      # AB[kd+i-j, j] = X[i, j], i <= j
    for d in range(1, kd + 1):                    # mirror: X[j+d, j] = X[j, j+d] = R_upper[kd-d, j+d]
        A[kd + d, : n - d] = R_upper[kd - d, d:]
    Cs = cinl.reshape(n, n1 * nl, order="F")
    G = self.dipole(A, Cs, Cs)
    return np.asfortranarray(G.reshape(n1, nl, n1, nl, order="F"))


BspAtom.TORMAT_RVEC = _tormat_rvec


def _dipole_chain(self, A_band: np.ndarray, C_blocks) -> np.ndarray:
    """D[l] = C[l+1]^T A C[l] for all neighbouring l in two launches (cfg5).  C_blocks: sequence of
    (n, nvec) arrays (e.g. BspAtom.cinl); returns (nl-1, nvec, nvec) with D[l] Fortran-ordered blocks."""
    A_band = np.asfortranarray(A_band, dtype=np.float64)
    nl = len(C_blocks)
    n, nvec = C_blocks[0].shape
    kd = (A_band.shape[0] - 1) // 2
    C_all = np.empty((nl, nvec, n))
    for l, Cm in enumerate(C_blocks):
        C_all[l] = np.asarray(Cm, dtype=np.float64).T      # block l column-major n x nvec
    D = np.empty((nl - 1, nvec, nvec))
    rc = self.lib.bspatom_dipole_chain(self._h, n, kd, A_band.ctypes.data_as(C.c_void_p), nl, nvec,
                                       C_all.ctypes.data_as(C.c_void_p), D.ctypes.data_as(C.c_void_p))
    _lib.check(self.lib, self._h, rc, "bspatom_dipole_chain")
    return np.transpose(D, (0, 2, 1))                       # D[l][f, i]


BspAtom.dipole_chain = _dipole_chain


def _dipole_chain_resident(self, A_band: np.ndarray, i0: int, nl: int, nvec: int) -> np.ndarray:
    """cfg5 on the eigenvectors the last batch left in HBM: D[l] = C[i0+l+1]^T A C[i0+l] (first nvec vectors each)."""
    A_band = np.asfortranarray(A_band, dtype=np.float64)
    kd = (A_band.shape[0] - 1) // 2
    D = np.empty((nl - 1, nvec, nvec))
    rc = self.lib.bspatom_dipole_chain_resident(self._h, int(i0), int(nl), int(nvec), kd,
                                                A_band.ctypes.data_as(C.c_void_p), D.ctypes.data_as(C.c_void_p))
    _lib.check(self.lib, self._h, rc, "bspatom_dipole_chain_resident")
    return np.transpose(D, (0, 2, 1))


def _wavefunction_resident(self, iprob: int, ivec0: int, nvec: int, ra: float, rb: float, npts: int = 10000):
    r = np.empty(npts + 1)
    psi = np.empty((npts + 1, nvec), order="F")
    rc = self.lib.bspatom_wavefunction_resident(self._h, int(iprob), int(ivec0), int(nvec), float(ra), float(rb), int(npts),
                                                r.ctypes.data_as(C.c_void_p), psi.ctypes.data_as(C.c_void_p))
    _lib.check(self.lib, self._h, rc, "bspatom_wavefunction_resident")
    return r, psi


BspAtom.dipole_chain_resident = _dipole_chain_resident
BspAtom.wavefunction_resident = _wavefunction_resident


class BspAtomMulti:
    """Several GPUs from one host process (bspatom_create_multi / bspatom_solve_batch_multi): what a single-process
    Fortran driver binds to spread the (instance, l) list of SOLVE_SYSTEM over the GPUs of a box (SURVEY.md 8(b)).
    bench.py uses one process per GPU instead; both shard the same way and neither has a collective on the compute path."""

    def __init__(self, devices: Sequence[int]):
        self.lib = _lib.load()
        self._m = C.c_void_p()
        ids = (C.c_int * len(devices))(*[int(d) for d in devices])
        rc = self.lib.bspatom_create_multi(C.byref(self._m), len(devices), ids)
        _lib.check(self.lib, None, rc, "bspatom_create_multi")
        self.devices = list(devices)

    def close(self):
        if getattr(self, "_m", None):
            self.lib.bspatom_destroy_multi(self._m)
            self._m = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name: str, value: float):
        if self.lib.bspatom_set_option_multi(self._m, name.encode(), float(value)):
            raise BspAtomError("bspatom_set_option_multi(%s) failed" % name)

    def solve_batch(self, items: Iterable, nvec: Optional[int] = None, select: Optional["Selection"] = None):
        """same contract as BspAtom.solve_batch: (list of E arrays, list of C blocks, info)"""
        items = list(items)
        arr, keep = build_problem_array(items, nvec, select)
        nfs, nvs = arr.rec["nfun"].astype(np.int64), arr.rec["nvec"].astype(np.int64)
        E, Cbuf = pinned_empty(int(nfs.sum())), pinned_empty(int((nfs * nvs).sum()))
        info = np.zeros(len(items), dtype=np.int32)
        rc = self.lib.bspatom_solve_batch_multi(self._m, len(items), arr, E.ctypes.data_as(C.c_void_p),
                                                Cbuf.ctypes.data_as(C.c_void_p), info.ctypes.data_as(_lib._ip))
        if rc:
            raise BspAtomError("bspatom_solve_batch_multi failed: rc=%d %s" % (rc, self.lib.bspatom_last_error_multi(self._m).decode()))
        eo = np.concatenate(([0], np.cumsum(nfs)))
        co = np.concatenate(([0], np.cumsum(nfs * nvs)))
        Es = [E[eo[i]:eo[i + 1]] for i in range(len(items))]
        Cs = [Cbuf[co[i]:co[i + 1]].reshape((int(nfs[i]), int(nvs[i])), order="F") for i in range(len(items))]
        return Es, Cs, info


class BspAtomPipeline:
    """Throughput mode for sweeps: `depth` handles on one GPU alternate over a list of batches, each from its
    own host thread (ctypes releases the GIL).  Every batch does its own H2D, kernels and D2H through
    `bspatom_solve_batch`; results land in the caller's (pinned) buffers.  The library sends the result copies
    of all handles through one FIFO queue per device, so the D2H of batch i (8 MB of eigenvectors per solve at
    N = 1000: the PCIe link is the longest leg) overlaps the kernels of batch i+1 and the sweep runs at the
    pace of the slower of the two legs.  Batches also take turns on the SMs (the library's per-device "compute
    turn"): started together they would only share the GPU and both finish late."""

    def __init__(self, device: int = 0, depth: int = 2):
        self.atoms = [BspAtom(device=device) for _ in range(depth)]
        self.batch_ms = None      # wall time of an undisturbed batch (fastest seen so far)
        self.timeline = []        # (batch, handle, start ms, end ms) of the last solve_batches call

    def set_option(self, name: str, value: float):
        for a in self.atoms:
            a.set_option(name, value)

    def close(self):
        for a in self.atoms:
            a.close()

    def solve_batches(self, batches, outs_E, outs_C, nvec=None, select=None, on_done=None):
        """batches[i]: list of (Problem, l); outs_E[i], outs_C[i]: pinned float64 buffers for batch i.
        select: device-side state selection applied to every batch; on_done(i, atom): called in the worker thread
        right after batch i returned (e.g. to read atom.selection() / atom.stats() of that batch).
        Returns the list of info arrays."""
        import threading
        import time

        infos = [None] * len(batches)
        errors = []
        took = []
        timeline = []
        t_origin = time.perf_counter()
        depth = len(self.atoms)
        stagger = 0.0   # the library's per-device compute turn orders the handles; no host-side delay needed

        def worker(w):
            try:
                if w and stagger > 0.0 and len(batches) > w:
                    time.sleep(w * stagger)
                for i in range(w, len(batches), depth):
                    t0 = time.perf_counter()
                    _, _, infos[i] = self.atoms[w].solve_batch(batches[i], nvec=nvec, out_E=outs_E[i], out_C=outs_C[i],
                                                               select=select)
                    if on_done is not None:
                        on_done(i, self.atoms[w])
                    t1 = time.perf_counter()
                    took.append(1e3 * (t1 - t0))
                    timeline.append((i, w, 1e3 * (t0 - t_origin), 1e3 * (t1 - t_origin)))
            except Exception as exc:       # surfaced to the caller below
                errors.append(exc)

        threads = [threading.Thread(target=worker, args=(w,)) for w in range(depth)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        self.timeline = sorted(timeline)
        if took:
            m = min(took)         # the least disturbed batch ~ one batch alone
            self.batch_ms = m if self.batch_ms is None else min(self.batch_ms, m)
        return infos


def pinned_empty(count: int) -> np.ndarray:
    """float64 array in page-locked host memory (bspatom_alloc_host): results written into it by
    solve_batch stream out chunk by chunk while the GPU keeps computing."""
    import weakref

    lib = _lib.load()
    nbytes = max(1, int(count)) * 8
    ptr = lib.bspatom_alloc_host(nbytes)
    if not ptr:
        raise BspAtomError("bspatom_alloc_host(%d bytes) failed" % nbytes)
    buf = (C.c_double * max(1, int(count))).from_address(ptr)
    arr = np.frombuffer(buf, dtype=np.float64, count=int(count))
    weakref.finalize(buf, lib.bspatom_free_host, ptr)
    return arr


def _to_c_problem(p: Problem, l: int, nvec: int, keep: list) -> BspProblem:
    cp = BspProblem()
    cp.k, cp.nfun, cp.nkp, cp.ka = int(p.k), int(p.nfun), int(p.nkp), int(p.ka)
    rt = np.ascontiguousarray(p.rt, dtype=np.float64)
    keep.append(rt)
    cp.rt = rt.ctypes.data_as(C.POINTER(C.c_double))
    if p.xg is not None:
        xg = np.ascontiguousarray(p.xg, dtype=np.float64)
        wg = np.ascontiguousarray(p.wg, dtype=np.float64)
        keep += [xg, wg]
        cp.xg = xg.ctypes.data_as(C.POINTER(C.c_double))
        cp.wg = wg.ctypes.data_as(C.POINTER(C.c_double))
    cp.pot_kind = int(p.pot_kind)
    par = list(p.pot_par) + [0.0] * 8
    for i in range(8):
        cp.pot_par[i] = float(par[i])
    if p.v_tab is not None:
        vt = np.ascontiguousarray(p.v_tab, dtype=np.float64)
        keep.append(vt)
        cp.v_tab = vt.ctypes.data_as(C.POINTER(C.c_double))
    cp.l = int(l)
    cp.ul_extra = float(p.bl[l]) if (p.bl is not None and p.pot_kind == POT_SIMONS_FUES) else 0.0
    cp.nvec = int(nvec)
    return cp


_PROBLEM_DTYPE = np.dtype({
    "names": ["k", "nfun", "nkp", "ka", "rt", "xg", "wg", "pot_kind", "pot_par", "v_tab", "l", "ul_extra", "nvec",
              "sel_mode", "sel_extra", "sel_group", "sel_ecut_a", "sel_ecut_b"],
    "formats": ["<i4", "<i4", "<i4", "<i4", "<u8", "<u8", "<u8", "<i4", ("<f8", 8), "<u8", "<i4", "<f8", "<i4",
                "<i4", "<i4", "<i4", "<f8", "<f8"],
    "offsets": [BspProblem.k.offset, BspProblem.nfun.offset, BspProblem.nkp.offset, BspProblem.ka.offset,
                BspProblem.rt.offset, BspProblem.xg.offset, BspProblem.wg.offset, BspProblem.pot_kind.offset,
                BspProblem.pot_par.offset, BspProblem.v_tab.offset, BspProblem.l.offset,
                BspProblem.ul_extra.offset, BspProblem.nvec.offset, BspProblem.sel_mode.offset,
                BspProblem.sel_extra.offset, BspProblem.sel_group.offset, BspProblem.sel_ecut_a.offset,
                BspProblem.sel_ecut_b.offset],
    "itemsize": C.sizeof(BspProblem),
})


@dataclass
class Selection:
    """Device-side state selection of SOLVE_SYSTEM's KIND_PI >= 3 branch (matrices.f90:296-334): keep the
    eigenvectors 1..ntemp, ntemp = MIN(MAX(n1_fin + 40, nlim), nfun).  Emax_fin / Elim as in the reference
    (Elim = Emax_fin + 0.25, or Emax_fin for KIND_PI >= 8); one running-maximum group per distinct Problem,
    its items in the order of the reference's l loop."""

    Emax_fin: float
    Elim: Optional[float] = None
    extra: int = 41          # n1_fin + 40 with n1_fin = count + 1

    @classmethod
    def from_kind_pi(cls, Emax_fin: float, kind_pi: int):
        return cls(Emax_fin, Emax_fin if kind_pi >= 8 else Emax_fin + 0.25)


def build_problem_array(items: List, nvec: Optional[int], select: Optional["Selection"] = None):
    """(Problem, l) list -> contiguous array of struct bsp_problem (numpy structured array with the
    C layout; filled per distinct Problem, not per item: a sweep has few instances and many l)."""
    keep: list = []
    n = len(items)
    rec = np.zeros(n, dtype=_PROBLEM_DTYPE)
    if select is not None:
        rec["sel_mode"] = 1
        rec["sel_extra"] = int(select.extra)
        rec["sel_ecut_a"] = float(select.Emax_fin)
        rec["sel_ecut_b"] = float(select.Emax_fin if select.Elim is None else select.Elim)
        gid, seen, last = np.zeros(n, dtype=np.int32), {}, None
        for i, (p, _) in enumerate(items):       # contiguous runs of one Problem form a group
            if last is None or id(p) != last:
                seen[i] = len(seen)
                cur = seen[i]
                last = id(p)
            gid[i] = cur
        rec["sel_group"] = gid
    groups: dict = {}
    for i, (p, l) in enumerate(items):
        groups.setdefault(id(p), (p, []))[1].append(i)
    ls = np.fromiter((l for _, l in items), dtype=np.int32, count=n)
    rec["l"] = ls
    for p, idx in groups.values():
        idx = np.asarray(idx)
        base = np.frombuffer(bytes(_to_c_problem(p, 0, 0, keep)), dtype=_PROBLEM_DTYPE, count=1)[0]
        for name in ("k", "nfun", "nkp", "ka", "rt", "xg", "wg", "pot_kind", "pot_par", "v_tab"):
            rec[name][idx] = base[name]
        rec["nvec"][idx] = p.nfun if nvec is None else min(int(nvec), p.nfun)
        if p.bl is not None and p.pot_kind == POT_SIMONS_FUES:
            rec["ul_extra"][idx] = np.asarray(p.bl, dtype=np.float64)[ls[idx]]
    keep.append(rec)
    arr = C.cast(rec.ctypes.data, C.POINTER(BspProblem))
    return _ProblemArray(arr, rec), keep


class _ProblemArray:
    """pointer to struct bsp_problem[] + the numpy record array that owns the memory"""

    def __init__(self, ptr, rec):
        self._as_parameter_ = ptr
        self.rec = rec

    def __getitem__(self, i):
        return self._as_parameter_[i]


def _band_operand(M, what: str):
    """(k+1, n) band in LAPACK storage -> (float64 array the pointer points into, leading dimension).  A Fortran-ordered
    float64 view with a longer column stride (AB = buf[:ka+1, :] of a (ldab, n) buffer) is passed as it is, with that
    stride as the leading dimension; anything else is copied into Fortran order."""
    M = np.asarray(M)
    if M.ndim != 2:
        raise ValueError("%s must be a 2-D band array of shape (k+1, n), got %d dimensions" % (what, M.ndim))
    if (M.dtype == np.float64 and M.strides[0] == 8 and M.shape[0] >= 1 and
            (M.shape[1] <= 1 or (M.strides[1] % 8 == 0 and M.strides[1] >= 8 * M.shape[0]))):
        return M, (M.strides[1] // 8 if M.shape[1] > 1 else M.shape[0])
    M = np.asfortranarray(M, dtype=np.float64)
    return M, max(1, M.shape[0])


def band_pencil_array(pencils: Iterable, nvec=None, uplo: str = "U"):
    """(AB, BB) / (AB, BB, uplo) list -> (struct bsp_band_pencil[], arrays it points into, n per pencil, nvec per
    pencil).  Operands that are not Fortran-ordered float64 are copied; the struct array holds a reference to every
    array it points into (a ctypes pointer stored in a struct does not keep its numpy array alive).  The half bandwidths are the band arrays' row counts minus one; the library checks their range, the
    leading dimensions, uplo's value and nvec.  nvec: None (every eigenvector), an int (capped at each n) or one
    value per pencil (passed as given)."""
    pens = list(pencils)
    if nvec is None or isinstance(nvec, (int, np.integer)):
        per = [None if nvec is None else int(nvec)] * len(pens)
        cap = True
    else:
        per = [int(v) for v in nvec]
        cap = False
        if len(per) != len(pens):
            raise ValueError("nvec has %d entries for %d pencils" % (len(per), len(pens)))
    arr = (BspBandPencil * max(1, len(pens)))()
    keep, ns, nvs = [], [], []
    for i, pen in enumerate(pens):
        if len(pen) not in (2, 3):
            raise ValueError("pencil %d: expected (AB, BB) or (AB, BB, uplo)" % i)
        up = pen[2] if len(pen) == 3 else uplo
        if not isinstance(up, str) or len(up) != 1:
            raise ValueError("pencil %d: uplo must be one character, 'U' or 'L'" % i)
        AB, ldab = _band_operand(pen[0], "AB")
        BB, ldbb = _band_operand(pen[1], "BB")
        if AB.shape[1] != BB.shape[1]:
            raise ValueError("pencil %d: AB has %d columns, BB %d" % (i, AB.shape[1], BB.shape[1]))
        n = AB.shape[1]
        nv = n if per[i] is None else (min(per[i], n) if cap else per[i])
        keep += [AB, BB]
        p = arr[i]
        p.n, p.ka, p.kb, p.uplo = n, AB.shape[0] - 1, BB.shape[0] - 1, up.encode()
        p.AB, p.ldab = AB.ctypes.data_as(C.POINTER(C.c_double)), ldab
        p.BB, p.ldbb = BB.ctypes.data_as(C.POINTER(C.c_double)), ldbb
        p.nvec = nv
        ns.append(n)
        nvs.append(nv)
    arr._keep = keep
    return arr, keep, ns, nvs


def dsbgv(AB: np.ndarray, BB: np.ndarray, jobz: str = "V", uplo: str = "U"):
    """LAPACK-shaped entry ``bspatom_dsbgv_``: A x = w B x for one band pencil, AB (ka+1, n) and BB (kb+1, n) in LAPACK
    band storage.  Returns (w, Z, info); Z is None for jobz = 'N'.  AB and BB are only read."""
    lib = _lib.load()
    A, ldab = _band_operand(AB, "AB")
    Bm, ldbb = _band_operand(BB, "BB")
    if A.shape[1] != Bm.shape[1]:
        raise ValueError("AB has %d columns, BB %d" % (A.shape[1], Bm.shape[1]))
    n = A.shape[1]
    wantz = jobz in ("V", "v")
    w = np.zeros(n)
    Z = np.zeros((n, n), order="F") if wantz else None      # not referenced for jobz = 'N'
    work = np.zeros(max(1, 3 * n))
    ci = lambda v: C.byref(C.c_int(v))
    info = C.c_int(0)
    lib.bspatom_dsbgv_(jobz.encode(), uplo.encode(), ci(n), ci(A.shape[0] - 1), ci(Bm.shape[0] - 1),
                       A.ctypes.data_as(C.c_void_p), ci(ldab), Bm.ctypes.data_as(C.c_void_p), ci(ldbb),
                       w.ctypes.data_as(C.c_void_p), Z.ctypes.data_as(C.c_void_p) if wantz else None,
                       ci(max(1, n) if wantz else 1),
                       work.ctypes.data_as(C.c_void_p), C.byref(info))
    return w, Z, info.value


def dsygv(H: np.ndarray, S: np.ndarray, jobz: str = "V", uplo: str = "U"):
    """LAPACK-shaped entry ``bspatom_dsygv_`` (the one-token rename of matrices.f90:248)."""
    lib = _lib.load()
    n = H.shape[0]
    A = np.asfortranarray(H, dtype=np.float64).copy(order="F")
    Bm = np.asfortranarray(S, dtype=np.float64).copy(order="F")
    w = np.zeros(n)
    work = np.zeros(max(1, 4 * n))
    ci = lambda v: C.byref(C.c_int(v))
    info = C.c_int(0)
    lib.bspatom_dsygv_(ci(1), jobz.encode(), uplo.encode(), ci(n), A.ctypes.data_as(C.c_void_p), ci(n),
                       Bm.ctypes.data_as(C.c_void_p), ci(n), w.ctypes.data_as(C.c_void_p),
                       work.ctypes.data_as(C.c_void_p), ci(4 * n), C.byref(info))
    return w, A, Bm, info.value
