"""GPU variant of tests/test_emul_rhs.py: the device's factor sweep (staged band tiles, cp.async look-ahead ring, FP64
FMA of sm_100a) forms S x and (H - rho S) x from the vector in X bit for bit in the order of the back sweep's column
sweep, at N = 1000 on cfg2-shaped pencils, for 1000 different vectors at once (one per eigen index)."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "emul", "gpu_rhs.cu")
dp = C.POINTER(C.c_double)


def upper_bands(A, B):
    n = A.shape[0]
    return np.ascontiguousarray(np.stack([np.r_[np.diag(A, d), np.zeros(d)] for d in range(B + 1)]))


@pytest.fixture(scope="module")
def gpu_rhs(tmp_path_factory):
    nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    so = str(tmp_path_factory.mktemp("gpu_rhs") / "libgpu_rhs.so")
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
                           "-Xcompiler", "-ffp-contract=off", "-shared", "-o", so, SRC])
    lib = C.CDLL(so)
    lib.gpu_rhs.argtypes = [C.c_int, dp, dp, dp, C.c_double, C.c_int, dp, dp]
    return lib


@pytest.mark.gpu
@pytest.mark.parametrize("l", [0, 50])
@pytest.mark.parametrize("resid", [0, 1], ids=["Sx", "H-rhoS"])
def test_device_formed_rhs_matches_column_sweep_bits_cfg2(gpu_rhs, l, resid):
    from oracle import oracle as O

    b = O.make_basis(kind_grid=0, k=7, nfun=1000, rb=500.0)
    m = O.matrix_svt(b, lmax=l, par=O.pot_params(0, 1.0 + 3 / 64.0))
    H = O.hamiltonian(m["T"], m["U"][:, :, l], m["V"])
    n, B = b.nfun, b.k - 1
    rng = np.random.default_rng(31 + l + resid)
    x = rng.standard_normal((n, n)) * np.exp(-np.linspace(0.0, 20.0, n))[None, :] ** rng.uniform(0, 1, (n, 1))
    x = np.ascontiguousarray(x)
    rho = -0.0123 if resid else 0.0
    hb, sb = upper_bands(H, B), upper_bands(m["S"], B)
    fused, ref = np.empty(n * n), np.empty(n * n)
    rc = gpu_rhs.gpu_rhs(n, hb.ctypes.data_as(dp), sb.ctypes.data_as(dp), x.ctypes.data_as(dp), rho, resid,
                         fused.ctypes.data_as(dp), ref.ctypes.data_as(dp))
    assert rc == 0
    seen = ~np.isnan(fused)
    assert seen.sum() >= n * (n // 2 - 7)
    assert np.array_equal(fused[seen].view(np.int64), ref[seen].view(np.int64))
