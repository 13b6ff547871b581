"""Shifted solves (H_l - z S) x = b on the benchmark's cfg2 step, in one command.

The step: 408 pencils, N = 1000 B-splines of order k = 7 on the linear grid (Rmax = 500), Coulomb Z = 1 + i/64 for
i = 0..7, l = 0..50, uploaded once (bspatom_batch_upload; no eigensolve).  128 shifts per pencil (52 224 systems),
nrhs = 1, B and X in device memory (torch tensors), real shifts spread over [-0.6, 3] and complex ones with
Im z in {1e-3, 1e-1}.  Reported per kind:

  systems_per_s       systems over the device ms the library reports for the call (CUDA events around its kernels)
  kernels             device ms per kernel name from torch.profiler (one profiled call, separate from the timed ones)
  bytes / GBs / frac  HBM bytes the kernels must move, from the shapes and the corrections the library counted
                      (bspatom_get_stats out[26]: their sum over all systems), over the device ms, and that rate as a
                      share of the device-to-device copy rate measured in the same run
  card                name and power limit, read in the same run

Prints one JSON object; writes nothing unless --out is given.
usage: python profiles/shifted_bench.py [--reps 5] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N, K, B, SHIFTS = 1000, 7, 6, 128


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    if q.returncode != 0:
        raise SystemExit("nvidia-smi failed: " + q.stderr)
    name, power, clock = [x.strip() for x in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def copy_peak_gbs(torch):
    """device-to-device copy of 4 GiB: bytes read + written over CUDA-event time, best of 5"""
    a = torch.empty(1 << 29, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 2 * a.numel() * 8 / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    del a, b
    torch.cuda.empty_cache()
    return best


def model_bytes(nsys, corrections, scalar):
    """HBM bytes of one call (nrhs = 1, every system solved).  A system that made k corrections ran k + 2 forward
    sweeps (step 0, then k + 1 that form the residual) and k + 1 back sweeps (step 0, then k that correct)."""
    s = 8 * scalar
    per_system = (2 * N * s + 2 * N * s      # b in (caller -> slots), x out (slots -> caller)
                  + N * (B + 1) * s          # factor written
                  + N * (B + 3) * s          # forward, step 0: L, b read, Y written
                  + N * (B + 4) * s          # the last forward sweep: L, b, x read, Y written
                  + N * (B + 2) * s)         # back, step 0: l, Y read, x written
    per_correction = N * (B + 4) * s + N * (B + 3) * s   # one more forward sweep and a correcting back sweep (x read)
    return nsys * per_system + corrections * per_correction


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    import bspatom_b200 as bsp
    from cases import host_basis

    a = host_basis(kind_grid=0, k=K, nfun=N, rb=500.0)
    items = []
    for iz in range(8):
        prob = bsp.Problem(k=a.k, nfun=a.nfun, nkp=a.nkp, ka=a.ka, rt=a.rt, pot_kind=bsp.POT_COULOMB, pot_par=(1.0 + iz / 64.0,))
        items += [(prob, l) for l in range(51)]
    npen = len(items)
    atom = bsp.BspAtom(device=0)
    atom.batch_upload(items, nvec=0)
    nsys = npen * SHIFTS
    iprob = np.repeat(np.arange(npen, dtype=np.int32), SHIFTS)
    zr = np.tile(np.linspace(-0.6, 3.0, SHIFTS) + 1.234e-5, npen)
    out = {"workload": "cfg2 step: %d pencils x %d shifts, N = %d, k = %d, nrhs = 1, B and X on the device" % (npen, SHIFTS, N, K),
           "card": card(), "copy_peak_GBs": copy_peak_gbs(torch)}
    g = torch.Generator(device="cuda").manual_seed(5)
    for kind in ("real", "complex"):
        cplx = kind == "complex"
        dt = torch.complex128 if cplx else torch.float64
        Bt = torch.randn(nsys * N, dtype=dt, device="cuda", generator=g)
        Xt = torch.empty_like(Bt)
        z = zr + 1j * np.tile(np.array([1e-3, 1e-1]), nsys // 2) if cplx else zr
        call = lambda: atom.shifted_solve_ptrs(iprob, z, 1, Bt.data_ptr(), Xt.data_ptr(), complex_=cplx)  # noqa: E731
        info, berr = call()    # warm-up (modules, workspace)
        ms, steps, corr = [], [], []
        for _ in range(args.reps):
            info, berr = call()
            st = atom.stats()
            ms.append(st["ms_shifted_solve"])
            steps.append(int(st["shifted_refinement_steps"]))
            corr.append(int(st["shifted_corrections"]))
        assert len(set(corr)) == 1 and np.all(info == 0)
        from torch.profiler import ProfilerActivity, profile

        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.events():
            if ev.device_type.name == "CUDA" and ("shifted" in ev.name or "combine" in ev.name):
                nm = ev.name.split("<")[0].split("(")[0].replace("void ", "")
                kern[nm] = kern.get(nm, 0.0) + getattr(ev, "device_time_total", 0.0) / 1e3
        dev_ms = float(np.median(ms))
        nbytes = model_bytes(nsys, corr[0], 2 if cplx else 1)
        gbs = nbytes / (dev_ms * 1e-3) / 1e9
        out[kind] = {"systems": nsys, "device_ms_median": dev_ms, "device_ms_all": ms, "systems_per_s": nsys / (dev_ms * 1e-3),
                     "corrections_max": max(steps), "corrections_total": corr[0],
                     "corrections_mean": corr[0] / nsys, "info_counts": {str(k): int(v) for k, v in zip(*np.unique(info, return_counts=True))},
                     "berr_max_solved": float(berr[info == 0].max()) if np.any(info == 0) else None,
                     "kernels_ms": kern, "bytes_model": nbytes, "GBs": gbs, "frac_of_copy_peak": gbs / out["copy_peak_GBs"]}
        del Bt, Xt
        torch.cuda.empty_cache()
    atom.close()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
