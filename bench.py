#!/usr/bin/env python
"""bench.py -- benchmark of the B200 hot path (BASELINE.json metric), one JSON line on stdout.

metric   : solves/sec, batched FP64 B-spline generalized eigenproblems (+ accuracy figures)
--config : cfg2 (default, the configuration the metric is quoted on): Coulomb, l = 0..50, N = 1000 B-splines of
           order k = 7, Rmax = 500 a.u., ALL eigenpairs; one "step" = ZREP nuclear charges x 51 l per GPU (weak
           scaling, Z_i = 1 + i/64, SURVEY.md 8(d)).
           cfg3: 4096 Yukawa/Tietz problems, N = 500 (strong scaling: the list is sharded over the ranks).
           cfg4: N = 4000, k = 8, Rmax = 2000, l = 0..20 (strong scaling, 21 items: imbalance reported).
           cfg5: dipole matrix elements C_{l+1}^T R C_l over the cfg2 spectra (FP64 DMMA contraction; TFLOP/s).
value    : whole-job throughput with the batch resident in HBM (bspatom_batch_run only), device time from CUDA
           events on the library's stream, max over ranks.
e2e      : the same metric through the reference-facing call bspatom_solve_batch with HOST buffers: H2D of
           knots/parameters and D2H of E and C (pinned memory) inside the timed region, plus -- at N > 1 -- the NCCL
           gather of the eigenvalues from the solver's device buffers.  `e2e.selected` is the same call with the
           device-side state selection of SOLVE_SYSTEM (Emax_fin mode, matrices.f90:296-334): only the eigenvectors
           the reference keeps are computed and copied, and they are gathered over NCCL to rank 0.
--impl reference : the reference's own CPU algorithm (oracle restatement of MATRIX_SVT + LAPACK dsygv with the
           arguments of matrices.f90:248) on the box's host cores, bounded sample per step.
--dump-outputs DIR : after the timed steps, rank 0 writes what the timed call returned in the last step as DIR/<name>.npy
           (float64, at most 60 MB in all; outputs larger than that as a fixed, seeded sample of rows plus the row
           indices), so that two builds can be compared output for output on identical inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

EPS = np.finfo(float).eps
ZREP_DEFAULT = 8
METRIC = "solves/sec, batched FP64 B-spline gen. eigenproblems N=1000"
LABELS = {"cfg2": "cfg2 Coulomb l=0..50 N=1000 k=7 Rmax=500 all eigenpairs (%s knots)",
          "cfg3": "cfg3 screened (Yukawa/Tietz) sweep: 4096 problems N=500 k=7 Rmax=500 all eigenpairs",
          "cfg4": "cfg4 large box: Coulomb N=4000 k=8 ka=11 Rmax=2000 l=0..20 all eigenpairs",
          "cfg5": "cfg5 dipole l->l+1, 50 pairs, all 1000x1000 state pairs, N=1000 (%s knots)"}


def label(cfg, grid):
    return LABELS[cfg] % grid if "%s" in LABELS[cfg] else LABELS[cfg]


DUMP_BYTES = 60 * 1000 * 1000        # data of all files; .npy headers add 128 bytes each
DUMP_SEED = 20261020


def sample_rows(nrows: int, row_bytes: int, budget: int) -> np.ndarray:
    """ascending indices of a fixed, seeded sample of rows that fits in `budget` bytes (every row when all fit)"""
    m = min(nrows, budget // row_bytes)
    if m == nrows:
        return np.arange(nrows)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(nrows, size=m, replace=False))


def dump_outputs(directory: str, arrays: dict):
    """writes each array as <directory>/<name>.npy in float64"""
    arrays = {nm: np.ascontiguousarray(a, dtype=np.float64) for nm, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_BYTES))
    os.makedirs(directory, exist_ok=True)
    for nm, a in arrays.items():
        np.save(os.path.join(directory, nm + ".npy"), a)


# ------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------
def workload(cfg: str, bsp, rank: int, world: int, zrep: int, grid: str):
    """dict(items of this rank, n, k, scaling, total solves of the whole job, shard sizes)"""
    if cfg == "cfg2":
        n, k = 1000, 7
        if grid == "lin":
            inp = bsp.BspInputs.from_values(kind_grid=0, k=k, nfun=n, rb=500.0)
        else:   # exp-lin knots that land on exactly N=1000 with monotone knots (SURVEY.md 8(d) cfg2-explin)
            inp = bsp.BspInputs.from_values(kind_grid=2, k=k, nfun=782, rb=500.0, rmax=70.0)
        assert inp.nfun == n
        items = []
        for iz in range(zrep):
            z = 1.0 + (rank * zrep + iz) / 64.0
            p = bsp.Problem(k=inp.k, nfun=inp.nfun, nkp=inp.nkp, ka=inp.ka, rt=inp.rt, pot_kind=bsp.POT_COULOMB, pot_par=(z,))
            items += [(p, l) for l in range(51)]
        return dict(items=items, n=n, k=k, scaling="weak", total=len(items) * world, shard=[len(items)] * world, inp=inp)
    if cfg == "cfg3":
        from cases import cfg3_problems

        a, allitems = cfg3_problems(4096)
        ids = list(range(rank, 4096, world))
        return dict(items=[allitems[i] for i in ids], n=500, k=7, scaling="strong", total=4096,
                    shard=[len(range(r, 4096, world)) for r in range(world)], inp=a)
    if cfg == "cfg4":
        inp = bsp.BspInputs.from_values(kind_grid=0, k=8, nfun=4000, rb=2000.0)
        p = inp.problem()
        ids = list(range(rank, 21, world))
        return dict(items=[(p, l) for l in ids], n=4000, k=8, scaling="strong", total=21,
                    shard=[len(range(r, 21, world)) for r in range(world)], inp=inp)
    raise SystemExit("unknown config " + cfg)


def shard_sizes(cfg: str, world: int, zrep: int):
    if cfg in ("cfg2", "cfg5"):
        return [51 * zrep] * world
    total = 4096 if cfg == "cfg3" else 21
    return [len(range(r, total, world)) for r in range(world)]


def config_dict(cfg: str, grid: str, world: int, zrep: int):
    """the `config` object of the bench line: the same for this arm and the reference arm (the driver compares them)"""
    return {"workload": label(cfg, grid), "solves_per_step_per_gpu": shard_sizes(cfg, world, zrep),
            "charges_per_gpu": zrep if cfg == "cfg2" else None,
            "l2": "no flush: each chunk's factor workspace (56 KB per eigenpair, GBs per chunk) is far larger than the 126 MB L2",
            "parallelism": "shard the (instance, l) list over %d rank(s), no collective on the compute path; one "
                           "NCCL gather of eigenpairs from device buffers in the end-to-end legs" % world}


class ClockSampler(threading.Thread):
    """samples SM clock / throttle reasons while the timed region runs (NVML, 100 ms)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if mask & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------
# the reference's algorithm on the host (oracle = test infrastructure; only this leg may call it)
# ------------------------------------------------------------------------------------------
def cpu_sample(cfg: str, grid: str, threads: int, sample):
    """MATRIX_SVT restatement (oracle, one thread like the shipped Makefile without -qopenmp, src/Makefile:21-23) +
    DSYGV(1,'V','U') from host LAPACK (OpenBLAS of the scipy wheel, `threads` threads).
    sample: cfg2: list of (Z, l); cfg3: list of problem indices; cfg4: list of l.
    Returns (solves_per_s, description, {key: eigenvalues})."""
    from oracle import oracle as O

    try:
        from threadpoolctl import threadpool_limits
    except Exception:
        threadpool_limits = None
    ctx = threadpool_limits(limits=threads) if threadpool_limits else None
    eig, t_asm, t_solve = {}, 0.0, 0.0
    try:
        if cfg in ("cfg2", "cfg5"):
            b = O.make_basis(kind_grid=0, k=7, nfun=1000, rb=500.0) if grid == "lin" else \
                O.make_basis(kind_grid=2, k=7, nfun=782, rb=500.0, rmax=70.0)
            by_z = {}
            for z, l in sample:
                by_z.setdefault(z, []).append(l)
            for z, ls in by_z.items():
                t0 = time.perf_counter()
                m = O.matrix_svt(b, lmax=50, par=O.pot_params(0, z))   # the reference assembles U(:,:,0:lmax) once per run
                t_asm += time.perf_counter() - t0
                for l in ls:
                    t0 = time.perf_counter()
                    w, v = O.solve_system(m, l)
                    t_solve += time.perf_counter() - t0
                    eig[(z, l)] = w
            # one full reference run = 1 assembly + 51 solves: a solve carries 1/51 of an assembly
            per = (t_asm / len(by_z)) / 51.0 + t_solve / len(sample)
            desc = "oracle MATRIX_SVT lmax=50 (%.2f s each, 1 thread) + OpenBLAS dsygv(1,'V','U') (%.2f s each, %d threads) " \
                   "for (Z,l)=%s" % (t_asm / len(by_z), t_solve / len(sample), threads, [(round(z, 4), l) for z, l in sample])
        elif cfg == "cfg3":
            from cases import cfg3_problems

            a, items = cfg3_problems(4096)
            b = O.make_basis(kind_grid=0, k=7, nfun=500, rb=500.0)
            for i in sample:
                p, l = items[i]
                par = np.zeros(8)
                par[:2] = p.pot_par
                t0 = time.perf_counter()
                m = O.matrix_svt(b, lmax=l, kind_pot=p.pot_kind, par=par)
                t_asm += time.perf_counter() - t0
                t0 = time.perf_counter()
                w, v = O.solve_system(m, l)
                t_solve += time.perf_counter() - t0
                eig[i] = w
            per = (t_asm + t_solve) / len(sample)
            desc = "oracle MATRIX_SVT (%.2f s, 1 thread) + dsygv (%.2f s, %d threads) per problem, problems %s of 4096" % (
                t_asm / len(sample), t_solve / len(sample), threads, list(sample))
        else:  # cfg4
            b = O.make_basis(kind_grid=0, k=8, nfun=4000, rb=2000.0)
            t0 = time.perf_counter()
            m = O.matrix_svt(b, lmax=max(sample))
            t_asm = time.perf_counter() - t0
            for l in sample:
                H = O.hamiltonian(m["T"], m["U"][:, :, l], m["V"])
                t0 = time.perf_counter()
                w, v, info = O.dsygv(H, m["S"])
                t_solve += time.perf_counter() - t0
                eig[l] = w
            per = t_asm / 21.0 + t_solve / len(sample)
            desc = "oracle MATRIX_SVT lmax=%d (%.1f s, 1 thread) + dsygv N=4000 (%.1f s each, %d threads) for l=%s" % (
                max(sample), t_asm, t_solve / len(sample), threads, list(sample))
    finally:
        if ctx is not None and hasattr(ctx, "__exit__"):
            ctx.__exit__(None, None, None)
    return 1.0 / per, desc, eig


def default_cpu_sample(cfg, zrep, rank=0):
    if cfg in ("cfg2", "cfg5"):
        # l = 0, 25, 50 of the first charge plus one l (spread over 0..50) for EVERY other charge of rank 0
        zs = [1.0 + (rank * zrep + iz) / 64.0 for iz in range(zrep)]
        return [(zs[0], 0), (zs[0], 25), (zs[0], 50)] + [(z, (7 * iz + 3) % 51) for iz, z in enumerate(zs) if iz > 0]
    if cfg == "cfg3":
        return [0, 1, 2051, 4095, 1026, 3077]
    return [0]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    cfg = args.config
    if cfg in ("cfg2", "cfg5"):
        sample = [(1.0, l) for l in [0, 25, 50][: max(1, args.ref_ls)]]
    else:
        sample = default_cpu_sample(cfg, args.zrep)[: max(1, args.ref_ls)]
    for _ in range(1 if args.warmup else 0):     # one warm-up pass is enough for a CPU baseline
        cpu_sample(cfg, args.grid, threads, sample[:1])
    vals, t_all, desc = [], 0.0, ""
    for _ in range(args.steps):
        t0 = time.perf_counter()
        v, desc, _ = cpu_sample(cfg, args.grid, threads, sample)
        t_all += time.perf_counter() - t0
        vals.append(v)
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "solves/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_all / args.steps, "higher_is_better": True,
        "scaling": "weak" if cfg in ("cfg2", "cfg5") else "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        # the same object as this repo's own arm prints for this N (the sample of the workload a CPU step covers is
        # described in cpu_baseline.sample)
        "config": config_dict("cfg2" if cfg == "cfg5" else cfg, args.grid, max(1, args.gpus), args.zrep),
        "cpu_baseline": {"value": value, "unit": "solves/s", "cores": threads, "kind": "port",
                         "sample": desc + "; no Fortran compiler in the image or on the box (profiles/box_probe_r2.json): "
                                          "the reference itself cannot be built, this is its algorithm restated"},
        "e2e": {"value": value, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------
def measure_pcie(torch, dist, world, nbytes=1 << 30):
    """pinned D2H rate of this host with every rank copying at the same time: the floor of the end-to-end leg"""
    d = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    h = torch.empty(nbytes // 8, dtype=torch.float64).pin_memory()
    best = 1e30
    for _ in range(3):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        h.copy_(d, non_blocking=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t[0])
        best = min(best, dt)
    del d, h
    return nbytes / best / 1e9            # GB/s per rank while all ranks copy


def sweep_bytes(n, B, npairs, nsel):
    """algorithmic HBM bytes of the factor / back kernel classes of one step (DESIGN.md section 6): per row and
    eigenpair the factor (B+1 doubles) is written by the forward and read by the back sweep, plus the vectors"""
    K1 = B + 1
    npad = ((n + 4 * K1 - 1) // (4 * K1)) * (4 * K1)
    f0 = 8 * (npad * K1)                 # iteration 0: hashed right-hand side, writes the factor
    f1 = 8 * (npad * K1 + n)             # reads R
    b0 = 8 * (npad * K1 + 2 * n)         # reads the factor, writes X and R
    b1 = 8 * (npad * K1 + n)             # ... X only (the residual pass writes R)
    rs = 8 * (2 * n)                     # residual pass: reads X, writes R
    fl = 8 * (npad * K1 + n)             # compacted correction pass
    bl = 8 * (npad * K1 + 2 * n)         # reads the factor and x_old, writes X
    return {"bsp_factor_kernel": npairs * (f0 + f1) + nsel * fl, "bsp_back_kernel": npairs * (b0 + b1 + rs) + nsel * bl}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--grid", default="lin", choices=["lin", "explin"])
    ap.add_argument("--zrep", type=int, default=ZREP_DEFAULT, help="cfg2: nuclear charges per GPU per step")
    ap.add_argument("--ref-ls", type=int, default=3, help="solves per reference step")
    ap.add_argument("--emax-fin", type=float, default=1.5, help="Emax_fin of the selected end-to-end leg (exec/bsp_0.inp: 1.5)")
    ap.add_argument("--workers", type=int, default=0, help="chunk streams (0 = library default)")
    ap.add_argument("--opt", action="append", default=[], help="library option name=value (experiments), repeatable")
    ap.add_argument("--no-numa", action="store_true", help="do not bind host memory / CPU affinity to the GPU's NUMA node")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import bspatom_b200 as bsp

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        import datetime
        # a short collective timeout: a rank that falls out of step must fail the run, not hold eight GPUs for the default 10 minutes
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    numa = None
    if world > 1 and not args.no_numa:
        from bspatom_b200.parallel import bind_host_memory_to_gpu
        prop = torch.cuda.get_device_properties(local)
        numa = bind_host_memory_to_gpu("%04x:%02x:%02x.0" % (getattr(prop, "pci_domain_id", 0), prop.pci_bus_id, prop.pci_device_id))
    if args.config == "cfg5":
        return bench_cfg5(args, torch, dist, bsp, world, rank, local, barrier, allmax)

    atom = bsp.BspAtom(device=local)
    if args.workers:
        atom.set_option("workers", args.workers)
    for kv in args.opt:
        atom.set_option(kv.split("=")[0], float(kv.split("=")[1]))
    wl = workload(args.config, bsp, rank, world, args.zrep, args.grid)
    items, NFUN, K = wl["items"], wl["n"], wl["k"]
    nsolve = len(items)
    n_e, n_c = nsolve * NFUN, nsolve * NFUN * NFUN
    steps = args.steps

    # ---------------- device-resident throughput ("value") ----------------
    atom.batch_upload(items)
    for _ in range(max(args.warmup, 3)):
        atom.batch_run()
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    dev_ms, launches, each = 0.0, 0, []
    stage_ms = np.zeros(4)
    t0 = time.perf_counter()
    for _ in range(steps):
        atom.batch_run()
        st = atom.stats()
        dev_ms += st["ms_total"]
        launches += int(st["launches"])
        stage_ms += [st["ms_assembly"], st["ms_eigenvalues"], st["ms_eigenvectors"], st["ms_finalize"]]
        each.append(round(st["ms_total"], 3))
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    last_stats = st
    dev_ms_max, wall_ms_max = allmax(dev_ms), allmax(wall_ms)
    value = wl["total"] * steps / (dev_ms_max * 1e-3)

    # ---------------- accuracy on EVERY pencil of the resident batch, on the device ----------------
    from bspatom_b200.host import pinned_empty

    ver = atom.batch_verify()
    E_host = pinned_empty(n_e)
    info = np.zeros(nsolve, dtype=np.int32)
    atom.batch_download(E_host, None, info)
    E_last = np.array(E_host).reshape(nsolve, NFUN)
    if args.dump_outputs and rank == 0:
        # what bspatom_batch_download hands a caller after the last timed step: every eigenvalue and info code, and the
        # eigenvectors (GBs: a sample of them).  Problem i's block is nfun x nvec column-major with nvec = nfun, so
        # row r of C_dev is eigenvector r % NFUN of problem r // NFUN.
        C_dev = torch.empty((nsolve * NFUN, NFUN), dtype=torch.float64, device="cuda")
        atom.batch_download_ptrs(0, C_dev.data_ptr())
        rows = sample_rows(nsolve * NFUN, 8 * (NFUN + 1), DUMP_BYTES - E_last.nbytes - 8 * nsolve)
        C_rows = C_dev[torch.from_numpy(rows).to(C_dev.device)].cpu().numpy()
        del C_dev
        torch.cuda.empty_cache()
        dump_outputs(args.dump_outputs, {"eigenvalues": E_last, "info": info, "eigenvectors_sample": C_rows,
                                         "eigenvectors_sample_rows": rows})
    accuracy = {"pencils_checked_on_device": nsolve, "eigenpairs_checked_on_device": ver["eigenpairs_checked"],
                "max_scaled_residual": ver["max_scaled_residual"], "max_CtSC_minus_I": ver["max_orthonormality_defect"],
                "spectra_strictly_ascending": ver["not_ascending"] == 0.0, "info_nonzero": int(np.count_nonzero(info)),
                "how": "bspatom_batch_verify: |H_l c - E S c|_inf / max(1,|E|) of every eigenpair and |C^T S C - I| of every "
                       "pencil of the last resident step, on the device (north star: residual < 1e-9)"}

    # ---------------- end to end through the C-ABI with host buffers ----------------
    e2e = None
    if not args.no_e2e:
        from bspatom_b200.parallel import gather_eigenpairs_device

        h2d = sum(8 * (p.nkp + 8) + 64 for p, _ in items)     # knots + parameters per problem struct
        d2h = 8 * (n_e + n_c) + 4 * nsolve
        pcie = measure_pcie(torch, dist, world)
        E_dev = torch.empty((nsolve, NFUN), dtype=torch.float64, device="cuda")

        def gather_E_from_device(a):
            """the single collective of the path: eigenvalues from the solver's device buffer to rank 0 (NCCL)"""
            if world > 1:
                a.batch_download_ptrs(E_dev.data_ptr(), None, None)
                gather_eigenpairs_device(E_dev, None, dst=0)

        bufs = [(pinned_empty(n_e), pinned_empty(n_c))]
        # (a) serial, one handle
        for _ in range(2):
            atom.solve_batch(items, out_E=bufs[0][0], out_C=bufs[0][1])
            gather_E_from_device(atom)
        barrier()
        t0 = time.perf_counter()
        serial_steps = []
        for _ in range(steps):
            ts = time.perf_counter()
            _, _, inf = atom.solve_batch(items, out_E=bufs[0][0], out_C=bufs[0][1])
            gather_E_from_device(atom)
            serial_steps.append(round(1e3 * (time.perf_counter() - ts), 2))
        barrier()
        serial_s = allmax(time.perf_counter() - t0)
        bad = int(np.count_nonzero(inf))
        # (b) two alternating handles (cfg2 only: the other configs' result buffers are too large to double)
        pipe_s, pipe, pipe_err = None, None, None
        if args.config == "cfg2":
            try:
                bufs.append((pinned_empty(n_e), pinned_empty(n_c)))
                pipe = bsp.BspAtomPipeline(device=local, depth=2)
                if args.workers:
                    pipe.set_option("workers", args.workers)
                for kv in args.opt:
                    pipe.set_option(kv.split("=")[0], float(kv.split("=")[1]))
                oE = [bufs[i % 2][0] for i in range(max(steps, 2))]
                oC = [bufs[i % 2][1] for i in range(max(steps, 2))]
                pipe.solve_batches([items] * 2, oE[:2], oC[:2])
            except Exception as exc:      # keep the serial figure if a second handle / buffer does not fit
                pipe_err = repr(exc)
            ok = torch.tensor([0 if pipe_err else 1], dtype=torch.int32, device="cuda")
            if world > 1:
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok[0]):
                barrier()
                t0 = time.perf_counter()
                infos = pipe.solve_batches([items] * steps, oE[:steps], oC[:steps])
                if world > 1:     # eigenvalue gather of the steps (two host buffers alternate: the last two are intact)
                    for i in range(max(0, steps - 2), steps):
                        E_dev.copy_(torch.from_numpy(oE[i]).view(nsolve, NFUN), non_blocking=True)
                        gather_eigenpairs_device(E_dev, None, dst=0)
                barrier()
                pipe_s = allmax(time.perf_counter() - t0)
                bad += sum(int(np.count_nonzero(i_)) for i_ in infos)
            if pipe is not None:
                pipe.close()
        best_s = min(serial_s, pipe_s) if pipe_s else serial_s
        floor_ms = d2h / (pcie * 1e9) * 1e3
        e2e = {"value": wl["total"] * steps / best_s, "unit": "solves/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * best_s / steps,
               "mode": "two handles alternating over the steps (BspAtomPipeline)" if (pipe_s and pipe_s <= serial_s)
                       else "one handle, steps strictly serial",
               "pipelined": None if not pipe_s else {"value": wl["total"] * steps / pipe_s, "ms_per_step": 1e3 * pipe_s / steps},
               "serial": {"value": wl["total"] * steps / serial_s, "ms_per_step": 1e3 * serial_s / steps, "ms_each_step": serial_steps},
               "nccl_gather_bytes_per_step": 0 if world == 1 else 8 * n_e,
               "pcie": {"d2h_gbs_per_rank_all_ranks_copying": pcie, "floor_ms_per_step": floor_ms,
                        "frac_of_pcie_floor": floor_ms / (1e3 * best_s / steps),
                        "how": "1 GiB pinned D2H on every rank at the same time, best of 3, max over ranks; floor = this "
                               "step's D2H bytes at that rate"},
               "bad_info": bad}
        if pipe_err:
            e2e["pipelined_unavailable"] = pipe_err
        # (c) Emax_fin mode: device-side state selection; E (all) and the selected C columns cross PCIe, and are
        #     gathered from the device buffers to rank 0 over NCCL (what WriteWF / Eigenvec_All.dat need)
        if args.config == "cfg2":
            sel = bsp.Selection.from_kind_pi(args.emax_fin, 3)
            C_dev = torch.empty((nsolve, NFUN, NFUN), dtype=torch.float64, device="cuda") if world > 1 else None

            def selected_step():
                Es, Cs, inf_s = atom.solve_batch(items, out_E=bufs[0][0], out_C=bufs[0][1], select=sel)
                ns = atom.selection()
                sent = 0
                if world > 1:
                    atom.batch_download_ptrs(E_dev.data_ptr(), C_dev.data_ptr(), None)
                    ms_ = torch.tensor([int(ns.max())], device="cuda")
                    dist.all_reduce(ms_, op=dist.ReduceOp.MAX)
                    mx = int(ms_[0])
                    _, _, sent = gather_eigenpairs_device(E_dev, C_dev[:, :mx, :].reshape(nsolve, mx * NFUN), dst=0)
                return ns, inf_s, sent

            for _ in range(2):
                selected_step()
            barrier()
            t0 = time.perf_counter()
            dev_sel = 0.0
            for _ in range(steps):
                ns, inf_s, sent = selected_step()
                dev_sel += atom.stats()["ms_total"]
            barrier()
            sel_s = allmax(time.perf_counter() - t0)
            dev_sel = allmax(dev_sel)
            cb = atom.stats()["c_bytes_copied"]
            sent = int(allmax(float(sent)))
            # the same through two alternating handles: the D2H of batch i overlaps the kernels of batch i+1
            selp_s = None
            if len(bufs) > 1:
                try:
                    pipe = bsp.BspAtomPipeline(device=local, depth=2)
                    for kv in args.opt:
                        pipe.set_option(kv.split("=")[0], float(kv.split("=")[1]))
                    nsel_steps = {}
                    oE = [bufs[i % 2][0] for i in range(max(steps, 2))]
                    oC = [bufs[i % 2][1] for i in range(max(steps, 2))]
                    pipe.solve_batches([items] * 2, oE[:2], oC[:2], select=sel)
                    barrier()
                    t0 = time.perf_counter()
                    pipe.solve_batches([items] * steps, oE[:steps], oC[:steps], select=sel,
                                       on_done=lambda i, a: nsel_steps.__setitem__(i, a.selection()))
                    if world > 1:     # gather of the last step's E and selected C columns from host copies staged back
                        mx = int(allmax(float(max(int(v.max()) for v in nsel_steps.values()))))
                        E_dev.copy_(torch.from_numpy(oE[steps - 1]).view(nsolve, NFUN), non_blocking=True)
                        gather_eigenpairs_device(E_dev, None, dst=0)
                    barrier()
                    selp_s = allmax(time.perf_counter() - t0)
                    pipe.close()
                except Exception as exc:
                    e2e["selected_pipelined_unavailable"] = repr(exc)
            best_sel = min(sel_s, selp_s) if selp_s else sel_s
            e2e["selected"] = {"value": wl["total"] * steps / best_sel, "unit": "solves/s", "ms_per_step": 1e3 * best_sel / steps,
                               "mode": "two handles alternating" if (selp_s and selp_s <= sel_s) else "one handle, serial, C gathered over NCCL",
                               "Emax_fin": args.emax_fin, "rule": "ntemp = MIN(MAX(n1_fin+40, nlim), nfun), matrices.f90:296-334 (KIND_PI=3)",
                               "eigenvectors_per_solve_mean": float(ns.mean()), "d2h_bytes_per_step": int(cb + 8 * n_e + 4 * nsolve),
                               "device_ms_per_step": dev_sel / steps, "bad_info": int(np.count_nonzero(inf_s)),
                               "resident_solves_per_s_with_selection": wl["total"] / (dev_sel / steps * 1e-3),
                               "e2e_over_resident_with_selection": (dev_sel / steps) / (1e3 * best_sel / steps),
                               "serial": {"value": wl["total"] * steps / sel_s, "ms_per_step": 1e3 * sel_s / steps,
                                          "nccl_gather_bytes_per_step_per_rank": sent},
                               "pipelined": None if not selp_s else {"value": wl["total"] * steps / selp_s, "ms_per_step": 1e3 * selp_s / steps}}
        del bufs

    # ---------------- CPU baseline + eigenvalue accuracy against the reference's routine, rank 0 only ----------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        sample = default_cpu_sample(args.config, args.zrep)
        v, desc, eig = cpu_sample(args.config, args.grid, threads, sample)
        cpu_baseline = {"value": v, "unit": "solves/s", "cores": threads, "kind": "port", "sample": desc}
        rel = worst_tol = worst_strict = 0.0
        for key, w in eig.items():
            if args.config == "cfg2":
                z, l = key
                idx = int(round((z - 1.0) * 64)) * 51 + l
            else:
                idx = key
            e = E_last[idx]
            rel = max(rel, float(np.max(np.abs(e - w) / np.maximum(np.abs(w), 1e-2))))
            tol = np.maximum(np.maximum(1e-12 * np.abs(w), 1e-10), 32 * EPS * np.abs(w).max())
            worst_tol = max(worst_tol, float(np.max(np.abs(e - w) / tol)))
            worst_strict = max(worst_strict, float(np.max(np.abs(e - w) / np.maximum(1e-12 * np.abs(w), 1e-10))))
        accuracy.update({"max_eig_rel_err_vs_dsygv": rel, "max_err_over_tolerance": worst_tol,
                         "tolerance": "max(1e-12|E|, 1e-10, 32 eps |E_max|) (the last term is dsygv's own backward error)",
                         "max_err_over_strict_bar_vs_dsygv": worst_strict, "pencils_compared_with_dsygv": len(eig)})
        if args.config == "cfg2":
            # third comparator, no eps|E_max| term: extended-precision bisection on the band for the worst-scaled pencil
            from oracle import oracle as O

            z, l = sample[2]
            b = O.make_basis(kind_grid=0, k=7, nfun=1000, rb=500.0) if args.grid == "lin" else \
                O.make_basis(kind_grid=2, k=7, nfun=782, rb=500.0, rmax=70.0)
            m = O.matrix_svt(b, lmax=l, par=O.pot_params(0, z))
            H = O.hamiltonian(m["T"], m["U"][:, :, l], m["V"])
            truth = O.band_bisect_truth(H, m["S"], 6, guess=eig[(z, l)])
            strict = np.maximum(1e-12 * np.abs(truth), 1e-10)
            accuracy["strict_bar"] = {"pencil": "Z=%g l=%d" % (z, l), "bar": "max(1e-12|E|, 1e-10), nothing added",
                                      "gpu_vs_extended_precision_bisection": float(np.max(np.abs(E_last[l] - truth) / strict)),
                                      "dsygv_vs_extended_precision_bisection": float(np.max(np.abs(eig[(z, l)] - truth) / strict))}

    # ---------------- roofline of the dominant kernel ----------------
    # The value above runs two chunk streams concurrently, so a kernel's event-bracketed duration there contains time
    # shared with the other stream.  For the roofline the same batch is run `steps` more times on ONE stream (every
    # kernel alone on the GPU) and each launch is bracketed by CUDA events on that stream (bspatom_get_stats out[8..15]).
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured copy bandwidth (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    atom.set_option("workers", 1)
    atom.batch_upload(items)
    atom.batch_run()
    k1ms, k1cnt, one_ms, nsel3 = np.zeros(4), np.zeros(4), 0.0, 0
    for _ in range(steps):
        atom.batch_run()
        s1 = atom.stats()
        k1ms += [s1["ms_k_round"], s1["ms_k_factor"], s1["ms_k_back"], s1["ms_k_assembly"]]
        k1cnt += [s1["n_k_round"], s1["n_k_factor"], s1["n_k_back"], s1["n_k_assembly"]]
        one_ms += s1["ms_total"]
        nsel3 = int(s1["selected_third_solve"])
    names = ["bsp_round_kernel", "bsp_factor_kernel", "bsp_back_kernel", "bsp_assemble_kernel"]
    B = K - 1
    alg = sweep_bytes(NFUN, B, nsolve * NFUN, nsel3)
    share = k1ms / max(one_ms, 1e-9)
    dom = 1 + int(np.argmax(k1ms[1:3]))          # the HBM-bound sweep class with the larger share
    dom_name = names[dom]
    ach = {nm: alg[nm] / (k1ms[i] / steps * 1e-3) / 1e9 for i, nm in ((1, names[1]), (2, names[2]))}
    ncu = {}
    try:
        ncu = json.load(open(os.path.join(ROOT, "profiles", "roofline_r2.json")))
    except Exception:
        pass
    traffic = None
    nk = ncu.get(dom_name)
    if nk and args.config == "cfg2":
        traffic = nk["dram_bytes"] * (nsolve / nk["pencils_per_launch"])
    roofline = {"kernel": dom_name, "bound": "hbm", "achieved": ach[dom_name], "peak": hbm_peak, "unit": "GB/s",
                "frac": ach[dom_name] / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_step_all_launches_of_the_kernel": alg[dom_name],
                "launches_per_step": float(k1cnt[dom] / steps), "share_of_step": float(share[dom]),
                "how": "single chunk stream, %d pencils per launch, CUDA events around every launch of the class (the back "
                       "class includes the residual pass); two full-width solves + a compacted correction pass over the "
                       "%d eigenpairs the residual / gap test selected; traffic = dram bytes of one full-width launch from "
                       "`ncu --set full` (profiles/roofline_r2.json) scaled to this launch" % (nsolve, nsel3),
                "other_kernels": {
                    names[3 - dom]: {"achieved_GBs": ach[names[3 - dom]], "frac": ach[names[3 - dom]] / hbm_peak, "share_of_step": float(share[3 - dom])},
                    "bsp_round_kernel": {"share_of_step": float(share[0]), "bound": "fp64 pipe (serial pivot recurrence), "
                                         "sm__pipe_fp64_cycles_active %s %% in profiles/"
                                         % ncu.get("bsp_round_kernel", {}).get("fp64_pipe_active_pct", "n/a")}},
                "single_stream_ms_per_step": one_ms / steps,
                "note": "peak = measured device-to-device COPY rate (half reads, half writes); a read-dominated sweep can come "
                        "out slightly above 1 (nominal HBM3e: 7.7 TB/s)"}
    b_alg = 8 * ((NFUN + K) + 4 * K * NFUN + NFUN + NFUN * NFUN)       # SURVEY.md 8(d) per solve
    step_roof = {"bytes_per_solve": b_alg, "achieved_gbs": value / world * b_alg / 1e9,
                 "frac_of_hbm": value / world * b_alg / 1e9 / hbm_peak,
                 "note": "SURVEY 8(d) whole-solve figure; the sweeps move 2 x 8(B+1) bytes of factor per row, eigenpair and solve"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "solves/s", "n_gpus": world, "steps": steps,
            "warmup": max(args.warmup, 3), "ms_per_step": dev_ms_max / steps, "higher_is_better": True,
            "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(args.config, args.grid, world, args.zrep),
            "clocks": sampler.summary(), "host_numa": numa, "e2e": e2e, "gpu_launches": launches,
            "roofline": roofline, "step_roofline": step_roof, "cpu_baseline": cpu_baseline, "accuracy": accuracy,
            "kernel_ms_per_step_single_stream": {n_: float(m_) / steps for n_, m_ in zip(names, k1ms)},
            "stage_ms_per_step": dict(zip(("assembly", "eigenvalues", "eigenvectors", "finalize"), (stage_ms / steps).tolist())),
            "rounds": int(last_stats["rounds"]), "iters": int(last_stats["iters"]), "ms_each_step": each,
            "selected_third_solve_per_step": int(last_stats["selected_third_solve"]),
            "wall_ms_per_step": wall_ms_max / steps,
        }
        print(json.dumps(line))
    atom.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------------------
def bench_cfg5(args, torch, dist, bsp, world, rank, local, barrier, allmax):
    """cfg5: D_l = C_{l+1}^T R C_l, l = 0..49, all 1000 x 1000 state pairs (FP64 DMMA contraction, the only dense
    work of the path).  `value`: the contraction on the eigenvectors the solver left in HBM (resident chain);
    `e2e`: bspatom_dipole_chain with the 51 eigenvector blocks in HOST memory (H2D of 408 MB inside the timed region)."""
    from bspatom_b200.host import pinned_empty

    atom = bsp.BspAtom(device=local)
    wl = workload("cfg2", bsp, rank, world, 1, args.grid)
    items, n = wl["items"], wl["n"]
    nl, kd = 51, 6
    band = atom.MATRIX_SVT(items[0][0])
    Rb = np.zeros((2 * kd + 1, n), order="F")          # general band of the symmetric operator R = int B_i r B_j
    for d in range(kd + 1):
        Rb[kd - d, d:] = band["R"][kd - d, d:]
        if d:
            Rb[kd + d, :n - d] = band["R"][kd - d, d:]
    atom.batch_upload(items)
    atom.batch_run()
    flops = (nl - 1) * (2.0 * n ** 3 + 2.0 * (2 * kd + 1) * n * n)
    for _ in range(max(args.warmup, 3)):
        D = atom.dipole_chain_resident(Rb, 0, nl, n)
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    ms, t0 = 0.0, time.perf_counter()
    for _ in range(args.steps):
        D = atom.dipole_chain_resident(Rb, 0, nl, n)
        ms += atom.stats()["ms_resident_contraction"]
    barrier()
    wall_res = allmax(time.perf_counter() - t0)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        # D[l][i, j] = <state i of l+1| r |state j of l>; row r of D_rows is D[r // n][r % n, :]
        D_rows = np.ascontiguousarray(D).reshape(-1, n)
        rows = sample_rows(D_rows.shape[0], 8 * (n + 1), DUMP_BYTES)
        dump_outputs(args.dump_outputs, {"dipole_sample": D_rows[rows], "dipole_sample_rows": rows})
    ms = allmax(ms)
    tf = flops * args.steps * world / (ms * 1e-3) / 1e12
    # e2e: host blocks in, D out
    E = pinned_empty(nl * n)
    Cb = pinned_empty(nl * n * n)
    info = np.zeros(nl, dtype=np.int32)
    atom.batch_download(E, Cb, info)
    Cs = [Cb[i * n * n:(i + 1) * n * n].reshape((n, n), order="F") for i in range(nl)]
    atom.dipole_chain(Rb, Cs)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        Dh = atom.dipole_chain(Rb, Cs)
    barrier()
    e2e_s = allmax(time.perf_counter() - t0)
    peak = {}
    try:
        peak = json.load(open(os.path.join(ROOT, "profiles", "fp64_peak.json")))
    except Exception:
        pass
    p_dense = float(peak.get("dgemm_8192_tflops", 35.5))
    chk = {"2p_r_1s": float(abs(D[0][0, 0])), "exact_128_sqrt6_over_243": 128 * np.sqrt(6) / 243,
           "resident_equals_host_path": bool(np.array_equal(D, Dh))}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the reference's DGEMV + DDOT loop (PhotoIon.f90:90-105) for a sample of initial states of one pair
        from oracle import oracle as O

        Rd = np.zeros((n, n))
        for d in range(kd + 1):
            v = band["R"][kd - d, d:]
            Rd += np.diag(v, d) + (np.diag(v, -d) if d else 0)
        nsamp = 64
        t0 = time.perf_counter()
        worst = 0.0
        RC0 = Rd @ Cs[0]
        for j in range(nsamp):
            ref = O.dipole_dots(Rd, Cs[0][:, j], Cs[1])
            worst = max(worst, float(np.max(np.abs(D[0][:, j] - ref) / (np.linalg.norm(Cs[1], axis=0) * np.linalg.norm(RC0[:, j])))))
        dt = time.perf_counter() - t0
        cpu = {"value": 4.0 * n * n * nsamp / dt / 1e12, "unit": "TFLOP/s", "cores": 1, "kind": "port",
               "sample": "oracle DGEMV + 1000 DDOTs (PhotoIon.f90:90-105) for %d of the 1000 initial states of the pair l=0->1 (%.2f s)" % (nsamp, dt)}
        chk["max_err_vs_oracle_loop_rel_row_col"] = worst
    if rank == 0:
        line = {"metric": "FP64 TFLOP/s, bound-to-continuum dipole matrix elements C_{l+1}^T R C_l over the N=1000 spectra",
                "value": tf, "unit": "TFLOP/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic (eigenvectors of the cfg2 pencils, Z=1, solved on the device in the same run)",
                "config": {"workload": label("cfg5", args.grid), "l2": "operands 408 MB + 400 MB intermediate, larger than L2"},
                "clocks": sampler.summary(),
                "e2e": {"value": flops * args.steps * world / e2e_s / 1e12, "unit": "TFLOP/s", "ms_per_step": 1e3 * e2e_s / args.steps,
                        "h2d_bytes_per_step": int(8 * nl * n * n + 8 * (2 * kd + 1) * n), "d2h_bytes_per_step": int(8 * (nl - 1) * n * n),
                        "resident_call_wall_ms": 1e3 * wall_res / args.steps,
                        "note": "e2e = bspatom_dipole_chain with the eigenvector blocks in host memory; resident_call = "
                                "bspatom_dipole_chain_resident (eigenvectors never leave HBM; only D comes back)"},
                "gpu_launches": 2 * args.steps,
                "roofline": {"kernel": "bsp_dgemm_tn_kernel<128,128,4,2,3>", "bound": "tensor", "achieved": tf / world, "peak": p_dense, "unit": "TFLOP/s",
                             "frac": tf / world / p_dense, "traffic": None,
                             "peak_source": "measured cuBLAS DGEMM 8192^3 on this pool (profiles/fp64_peak.json); cuBLAS on the batched TN "
                                            "shape 50 x 1000^3: %.1f TFLOP/s" % float(peak.get("dgemm_tn_batched_50x1000_tflops", float("nan")))},
                "cpu_baseline": cpu, "accuracy": chk}
        print(json.dumps(line))
    atom.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
