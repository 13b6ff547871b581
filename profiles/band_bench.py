"""Caller-supplied band pencils against the assembled path on the benchmark's cfg2 step, in one command.

The step: 408 pencils, N = 1000 B-splines of order k = 7 on the linear grid (Rmax = 500), Coulomb Z = 1 + i/64 for
i = 0..7, l = 0..50.  The band inputs are bspatom_assemble_band's S and H_l = H0 + l(l+1) Q formed on the host, so both
paths solve the same pencils.  Two handles keep one batch resident each; the measurements alternate between them:

  resident      host wall ms of bspatom_batch_run (ends in a stream synchronise) per step: the assembled path
                (bspatom_batch_upload once, then run: assembly + solver) against the band path (bspatom_band_upload
                once, then run: solver only), and the device ms the library reports for the run
  band_upload   host wall ms of bspatom_band_upload: checks and packing on the host, one H2D copy, ingest and the
                positive-definiteness check of B
  e2e           host wall ms of bspatom_solve_band_batch into pinned buffers (upload + run + streamed D2H)
  dsygv         host wall ms of bspatom_dsygv_ per pencil (dense N x N input), over a few pencils, for scale

Prints one JSON object with the card name and power limit read in the same run.  Writes nothing unless --out is given.
usage: python profiles/band_bench.py [--reps 20] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    if q.returncode != 0:
        raise SystemExit("nvidia-smi failed: " + q.stderr)
    name, power, clock = [x.strip() for x in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def summary(xs):
    return {"median_ms": statistics.median(xs), "min_ms": min(xs), "max_ms": max(xs), "n": len(xs)}


def wall(f):
    t0 = time.perf_counter()
    f()
    return 1e3 * (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import bspatom_b200 as bsp
    from bspatom_b200.host import pinned_empty

    dev = card()
    inp = bsp.BspInputs.from_values(kind_grid=0, k=7, nfun=1000, rb=500.0)
    n = inp.nfun
    probs = [bsp.Problem(k=inp.k, nfun=n, nkp=inp.nkp, ka=inp.ka, rt=inp.rt, pot_kind=bsp.POT_COULOMB, pot_par=(1.0 + i / 64.0,))
             for i in range(8)]
    items = [(p, l) for p in probs for l in range(51)]
    asm, band = bsp.BspAtom(device=0), bsp.BspAtom(device=0)
    bands = [band.MATRIX_SVT(p) for p in probs]
    pens = [(np.asfortranarray(b["H0"] + (l * (l + 1)) * b["Q"]), b["S"]) for b in bands for l in range(51)]
    npen = len(pens)
    asm.batch_upload(items)
    band.band_upload(pens)
    for h in (asm, band):       # warm-up: modules, workspaces, helper streams
        h.batch_run()
        h.batch_run()
    # same answer: the band path solves the pencils the assembled path assembles (H_l rounded differently: tolerance)
    Ea, Eb = np.empty(npen * n), np.empty(npen * n)
    ia, ib = np.zeros(npen, np.int32), np.zeros(npen, np.int32)
    asm.batch_download(Ea, None, ia)
    band.batch_download(Eb, None, ib)
    assert not ia.any() and not ib.any()
    max_rel_e = float(np.max(np.abs(Ea - Eb) / np.maximum(1.0, np.abs(Ea))))
    res = {"asm": [], "band": [], "asm_dev": [], "band_dev": [], "upload": [], "e2e": []}
    for _ in range(args.reps):
        res["asm"].append(wall(asm.batch_run))
        res["asm_dev"].append(asm.stats()["ms_total"])
        res["band"].append(wall(band.batch_run))
        res["band_dev"].append(band.stats()["ms_total"])
    ver = band.batch_verify()
    pE, pC = pinned_empty(npen * n), pinned_empty(npen * n * n)
    band.solve_band_batch(pens, out_E=pE, out_C=pC)           # warm-up of the streamed geometry
    for _ in range(max(3, args.reps // 4)):
        res["upload"].append(wall(lambda: band.band_upload(pens)))
        res["e2e"].append(wall(lambda: band.solve_band_batch(pens, out_E=pE, out_C=pC)))
    # the single-pencil LAPACK-shaped entry, dense input, for scale
    from cases import band_to_dense_sym

    dsy = []
    for b, l in ((bands[0], 0), (bands[3], 25), (bands[7], 50), (bands[0], 1), (bands[5], 10)):
        H = band_to_dense_sym(b["H0"] + (l * (l + 1)) * b["Q"], n)
        S = band_to_dense_sym(b["S"], n)
        bsp.dsygv(H, S)                                          # first call creates the shared handle
        dsy.append(wall(lambda: bsp.dsygv(H, S)))
    out = {
        "card": dev, "step": "cfg2 lin: %d pencils N=%d k=7 (l=0..50 x 8 charges)" % (npen, n),
        "resident_wall_ms": {"assembled": summary(res["asm"]), "band": summary(res["band"])},
        "resident_device_ms": {"assembled": summary(res["asm_dev"]), "band": summary(res["band_dev"])},
        "band_over_assembled_resident": statistics.median(res["band"]) / statistics.median(res["asm"]),
        "band_upload_wall_ms": summary(res["upload"]),
        "band_e2e_pinned_wall_ms": summary(res["e2e"]),
        "band_e2e_solves_per_s": npen / (statistics.median(res["e2e"]) * 1e-3),
        "dsygv_per_pencil_wall_ms": summary(dsy),
        "band_verify": ver, "max_rel_diff_E_band_vs_assembled": max_rel_e,
    }
    txt = json.dumps(out)
    print(txt)
    if args.out:
        with open(args.out, "w") as f:
            f.write(txt + "\n")
    asm.close()
    band.close()


if __name__ == "__main__":
    main()
