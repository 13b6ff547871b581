"""GPU: one answer, whichever path delivers it.  The cfg2 step as the benchmark runs it (linear knots, N = 1000, k = 7,
Rmax = 500, Coulomb Z = 1 + i/64 for i = 0..7, l = 0..50: 408 pencils) solved resident, checked on its own, and then
through every path that streams, pipelines, shards or redoes it: DESIGN.md section 9 promises the same bits however a
work list is chunked or sharded.

Streamed results cut the batch into chunks of shrinking size on two chunk streams and copy each chunk out through the
per-device copy queue as soon as it is final; a chunk that runs out of bracketing rounds or refinement iterations is
redone with the full limits and copied again.  So that stale data cannot pass, every pinned output buffer is filled
with NaN before a call, and the handle solves a different workload (other charges) right before the call under test."""
import re

import numpy as np
import pytest

import bspatom_b200 as bsp
from bspatom_b200 import postproc
from bspatom_b200.host import pinned_empty
from cases import check_eigenpairs, eig_tolerance, host_basis

pytestmark = pytest.mark.gpu

N, LS = 1000, range(51)
ZS = [1.0 + i / 64.0 for i in range(8)]
ZS_OTHER = [2.0 + i / 64.0 for i in range(8)]
SEL = bsp.Selection.from_kind_pi(1.5, 3)          # Emax_fin of the shipped input, KIND_PI = 3
DEFAULTS = {"rounds_enqueued": 26, "max_rounds": 90, "stream_chunks": 6, "stream_workers": 2, "workers": 2, "chunk": 0,
            "trace": 0}


def cfg2_items(zs, ls=LS, nfun=N):
    a = host_basis(kind_grid=0, k=7, nfun=nfun, rb=500.0 if nfun == N else 150.0)
    items = []
    for z in zs:
        p = bsp.Problem(k=a.k, nfun=a.nfun, nkp=a.nkp, ka=a.ka, rt=a.rt, pot_kind=bsp.POT_COULOMB, pot_par=(z,))
        items += [(p, l) for l in ls]
    return items


ITEMS, OTHER = cfg2_items(ZS), cfg2_items(ZS_OTHER)
NE, NC = N * len(ITEMS), N * N * len(ITEMS)


class options:
    """set options on a handle (BspAtom, BspAtomMulti, BspAtomPipeline) and put the defaults back on exit"""

    def __init__(self, h, **kw):
        self.h, self.kw = h, kw

    def __enter__(self):
        for k, v in self.kw.items():
            self.h.set_option(k, v)

    def __exit__(self, *exc):
        for k in self.kw:
            self.h.set_option(k, DEFAULTS[k])


def resident(h, items, select=None, vectors=True):
    """batch_upload + batch_run + batch_download into fresh NaN buffers"""
    h.batch_upload(items, select=select)
    h.batch_run()
    E, Cb, info = np.full(NE, np.nan), np.full(NC, np.nan) if vectors else None, np.full(len(items), -1, np.int32)
    h.batch_download(E, Cb, info)
    return E, Cb, info


def scramble(h):
    """solve another workload of the same shapes on h: device buffers no longer hold the answer under test"""
    h.batch_upload(OTHER)
    h.batch_run()


@pytest.fixture(scope="module")
def ref(atom):
    E, Cb, info = resident(atom, ITEMS)
    st, ver = atom.stats(), atom.batch_verify()
    Es, Cs, info_s = resident(atom, ITEMS, select=SEL)
    nsel = atom.selection()
    E_other = resident(atom, OTHER, vectors=False)[0]
    return dict(E=E, C=Cb, info=info, stats=st, verify=ver, E_sel=Es, C_sel=Cs, info_sel=info_s, nsel=nsel,
                E_other=E_other)


@pytest.fixture(scope="module")
def pinned():
    return [(pinned_empty(NE), pinned_empty(NC)) for _ in range(2)]


def nan_fill(*bufs):
    for b in bufs:
        b.fill(np.nan)


def assert_same(E, Cb, info, ref):
    assert np.array_equal(np.asarray(info), ref["info"]) and not ref["info"].any()
    assert np.array_equal(E, ref["E"])
    assert np.array_equal(Cb, ref["C"])


def assert_same_selected(E, Cb, info, nsel, ref):
    """E bit-identical to the selected resident run, the same counts, the first nsel columns of every block bit-identical"""
    assert not np.asarray(info).any() and np.array_equal(nsel, ref["nsel"])
    assert np.array_equal(E, ref["E_sel"])
    for i, k in enumerate(nsel):
        blk = slice(i * N * N, i * N * N + k * N)       # column-major: the first k columns are a prefix of the block
        assert np.array_equal(Cb[blk], ref["C_sel"][blk]), i


def test_reference_run_checks_out(ref, oracle):
    """the resident run is what the other paths are compared with, so it is checked independently: batch_verify over
    every pencil, and three pencils against the oracle (extended-precision bisection on the band, oracle-assembled H, S)"""
    from test_gpu_solve import oracle_pencil, strict_tolerance

    v = ref["verify"]
    assert v["eigenpairs_checked"] == len(ITEMS) * N
    assert v["max_scaled_residual"] <= 1e-11 and v["max_orthonormality_defect"] <= 1e-10 and v["not_ascending"] == 0.0
    assert not ref["info"].any()
    a = host_basis(kind_grid=0, k=7, nfun=N, rb=500.0)
    for z, l in ((1.0, 0), (1.109375, 25), (1.0, 50)):
        i = ZS.index(z) * len(LS) + l
        E = ref["E"][i * N:(i + 1) * N]
        Cm = ref["C"][i * N * N:(i + 1) * N * N].reshape((N, N), order="F")
        b, H, S = oracle_pencil(oracle, a, N, l, par=oracle.pot_params(0, z))
        w, _, _ = oracle.dsygv(H, S)
        truth = oracle.band_bisect_truth(H, S, 6, guess=w)
        assert np.all(np.abs(E - truth) <= strict_tolerance(truth)), (z, l)
        check_eigenpairs(E, Cm, H, S, res_tol=1e-11, orth_tol=1e-10)


def test_streamed_default(atom, ref, pinned):
    E, Cb = pinned[0]
    scramble(atom)
    nan_fill(E, Cb)
    _, _, info = atom.solve_batch(ITEMS, out_E=E, out_C=Cb)
    assert_same(E, Cb, info, ref)


@pytest.mark.parametrize("opt", [{"stream_workers": 1}, {"stream_chunks": 3}])
def test_streamed_other_geometries(atom, ref, pinned, opt):
    E, Cb = pinned[0]
    scramble(atom)
    nan_fill(E, Cb)
    with options(atom, **opt):
        _, _, info = atom.solve_batch(ITEMS, out_E=E, out_C=Cb)
    assert_same(E, Cb, info, ref)


@pytest.mark.parametrize("opt", [{"workers": 1}, {"chunk": 37}])
def test_resident_other_geometries(atom, ref, opt):
    """one chunk stream; chunks of 37 pencils (the last one ragged)"""
    scramble(atom)
    with options(atom, **opt):
        E, Cb, info = resident(atom, ITEMS)
    assert_same(E, Cb, info, ref)


def run_pipeline(ref, pinned, select=None):
    """BspAtomPipeline(depth=2) over [this workload, the other one, this workload]: batches 0 and 2 run on the same
    handle into the same buffers, checked (and refilled with NaN) as each batch returns"""
    batches = [ITEMS, OTHER, ITEMS]
    oE, oC = [pinned[0][0], pinned[1][0], pinned[0][0]], [pinned[0][1], pinned[1][1], pinned[0][1]]
    nan_fill(*pinned[0], *pinned[1])
    checked = []

    def on_done(i, h):
        E, Cb = oE[i], oC[i]
        if i == 1:
            assert np.isfinite(E).all()
            if select is None:
                assert np.array_equal(E, ref["E_other"])
        elif select is None:
            assert_same(E, Cb, np.zeros(len(ITEMS), np.int32), ref)
        else:
            nsel = h.selection()
            assert_same_selected(E, Cb, np.zeros(len(ITEMS), np.int32), nsel, ref)
            assert h.stats()["c_bytes_copied"] == 8 * N * int(nsel.sum())
        checked.append(i)
        nan_fill(E, Cb)

    pipe = bsp.BspAtomPipeline(device=0, depth=2)
    try:
        infos = pipe.solve_batches(batches, oE, oC, select=select, on_done=on_done)
    finally:
        pipe.close()
    assert sorted(checked) == [0, 1, 2]
    assert not any(i.any() for i in infos)


def test_pipeline(ref, pinned):
    run_pipeline(ref, pinned)


def test_multi_two_handles_one_device(ref):
    multi = bsp.BspAtomMulti([0, 0])
    try:
        multi.solve_batch(OTHER)
        Es, Cs, info = multi.solve_batch(ITEMS)
    finally:
        multi.close()
    assert np.array_equal(info, ref["info"])
    assert np.array_equal(np.concatenate(Es), ref["E"])
    for i, c in enumerate(Cs):
        assert np.array_equal(c.ravel(order="F"), ref["C"][i * N * N:(i + 1) * N * N]), i


def test_selected_streamed_and_pipelined(atom, ref, pinned):
    """Emax_fin mode: the device keeps the eigenvectors 1..ntemp of the reference's l loop (matrices.f90:296-334)"""
    Enl = ref["E_sel"].reshape(len(ZS), len(LS), N)
    want = np.concatenate([postproc.select_states(Enl[iz].T, 3, 0, LS[-1], SEL.Emax_fin).ntemp for iz in range(len(ZS))])
    assert np.array_equal(ref["nsel"], want) and not ref["info_sel"].any()
    assert ref["nsel"].max() < N
    E, Cb = pinned[0]
    scramble(atom)
    nan_fill(E, Cb)
    _, _, info = atom.solve_batch(ITEMS, out_E=E, out_C=Cb, select=SEL)
    nsel = atom.selection()
    assert_same_selected(E, Cb, info, nsel, ref)
    assert atom.stats()["c_bytes_copied"] == 8 * N * int(nsel.sum())
    run_pipeline(ref, pinned, select=SEL)


TRACE = re.compile(r"\[bspatom trace \S+\] chunk (\d+) stream (\d+) pencils (\d+) ")


def traced_geometry(atom, ref, pinned, capfd):
    """(chunk, stream, pencils) of the streamed cfg2 step, from the trace of one run (trace copies each chunk through its
    own path, so the bit-identity tests run without it)"""
    E, Cb = pinned[0]
    nan_fill(E, Cb)
    capfd.readouterr()
    with options(atom, trace=1):
        _, _, info = atom.solve_batch(ITEMS, out_E=E, out_C=Cb)
    chunks = [tuple(int(x) for x in m.groups()) for m in TRACE.finditer(capfd.readouterr().err)]
    assert_same(E, Cb, info, ref)
    return chunks


def test_streamed_geometry(atom, ref, pinned, capfd):
    """what the tests above claim to cover: at least 4 chunks of non-increasing size on 2 streams, 408 pencils in all"""
    chunks = traced_geometry(atom, ref, pinned, capfd)
    sizes = [n for _, _, n in sorted(chunks)]
    assert len(chunks) >= 4 and sum(sizes) == len(ITEMS), chunks
    assert all(a >= b for a, b in zip(sizes, sizes[1:])), chunks
    assert len({w for _, w, _ in chunks}) == 2, chunks


def test_redo_path(atom, ref, pinned, capfd):
    """rounds_enqueued = 1: every chunk hands over crowded brackets and is redone with max_rounds / max_iters, resident,
    streamed (the redo copies the chunk again behind its first copy) and through BspAtomMulti.  Surplus launches return
    at once, so the redone chunks give the reference's bits as long as the reference stayed inside the enqueued
    schedule (rounds < 26, iterations < 5).  The selected mode cannot be forced into a redo by options: its bracketing
    enqueues at least 64 rounds whatever rounds_enqueued says."""
    assert ref["stats"]["rounds"] < 26 and ref["stats"]["iters"] < 5, ref["stats"]
    n_streamed = len(traced_geometry(atom, ref, pinned, capfd))
    scramble(atom)
    with options(atom, rounds_enqueued=1):
        E, Cb, info = resident(atom, ITEMS)
        assert atom.stats()["chunks_redone"] == 2          # two equal chunks, one per chunk stream
        assert_same(E, Cb, info, ref)
        E, Cb = pinned[0]
        scramble(atom)
        nan_fill(E, Cb)
        _, _, info = atom.solve_batch(ITEMS, out_E=E, out_C=Cb)
        assert atom.stats()["chunks_redone"] == n_streamed >= 2
        assert_same(E, Cb, info, ref)
    multi = bsp.BspAtomMulti([0, 0])
    try:
        multi.solve_batch(OTHER)
        multi.set_option("rounds_enqueued", 1)
        Es, Cs, info = multi.solve_batch(ITEMS)
    finally:
        multi.close()
    assert np.array_equal(info, ref["info"])
    assert np.array_equal(np.concatenate(Es), ref["E"])
    for i, c in enumerate(Cs):
        assert np.array_equal(c.ravel(order="F"), ref["C"][i * N * N:(i + 1) * N * N]), i


def test_exhausted_budget_is_reported(atom, oracle):
    """max_rounds = 2 caps the bracketing (rounds_enqueued too) and the redo cannot do better: the call returns, and every
    pencil whose eigenvalues or eigenpairs are wrong says so in info (include/bspatom.h: info reports the affected
    pencils rather than returning wrong eigenpairs silently)"""
    from test_gpu_solve import oracle_pencil

    n, items = 300, cfg2_items([1.0], range(6), nfun=300)
    a = host_basis(kind_grid=0, k=7, nfun=n, rb=150.0)
    E0, C0, info0 = atom.solve_batch(items)
    assert not info0.any()
    pencils = [oracle_pencil(oracle, a, n, l)[1:] for l in range(6)]
    with options(atom, max_rounds=2):
        runs = {"streamed": atom.solve_batch(items)}
        atom.batch_upload(items)
        atom.batch_run()
        E, Cb, info = np.empty(6 * n), np.empty(6 * n * n), np.zeros(6, np.int32)
        atom.batch_download(E, Cb, info)
        runs["resident"] = ([E[i * n:(i + 1) * n] for i in range(6)],
                            [Cb[i * n * n:(i + 1) * n * n].reshape((n, n), order="F") for i in range(6)], info)
    wrong_seen = 0
    for how, (Es, Cs, info) in runs.items():
        for l, ((H, S), E, Cm) in enumerate(zip(pencils, Es, Cs)):
            wrong = not np.all(np.abs(E - E0[l]) <= eig_tolerance(E0[l]))
            try:
                check_eigenpairs(E, Cm, H, S)
            except AssertionError:
                wrong = True
            wrong_seen += wrong
            assert not wrong or info[l] != 0, (how, l)
    print("max_rounds = 2: %d of 12 pencils wrong, all reported" % wrong_seen)
