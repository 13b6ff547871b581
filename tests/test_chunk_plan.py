"""How the batch runner cuts a group of pencils into chunks (bsp_plan_chunks, bspatom_b200/csrc/bsp_plan.h).

The plan sets the streamed end-to-end rate (DESIGN.md section 5) and decides which chunkings the bit-identity promise
covers (section 9).  The header includes nothing from CUDA, so this test compiles it with g++ through
tests/emul/emul_plan.cpp and needs no GPU.  The golden table was recorded from the planning code as it stood inside
the runner before it moved into the header.

Three properties the sweep pins are looser than they may look.  A shrinking cut sizes its chunks from the cap on
average, so its first chunk can exceed the cap by the factor (nchunks + 2) / nchunks.  In a batch of a few pencils per
chunk, the rounding of a bound can make a chunk one pencil larger than the one before it.  And moving bounds to the ends
of selection groups can push a chunk over the cap even when every group fits it; the runner then refuses the batch
just as it does for a group that is too large on its own."""
import ctypes as C
import os
import random
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "emul", "emul_plan.cpp")
ip = C.POINTER(C.c_int)
BIG = 1 << 24                                    # budget that does not bind
SEL51 = [(1, i // 51) for i in range(408)]       # the cfg2 selection batch: 8 groups of 51 pencils
SEL30 = [(1, i // 30) for i in range(408)]


@pytest.fixture(scope="module")
def plan(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emul_plan") / "libemul_plan.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, SRC])
    lib = C.CDLL(so)
    lib.emul_plan.argtypes = [C.c_int] * 8 + [ip, ip, ip, ip, ip]
    lib.emul_plan.restype = C.c_int

    def run(npencil, n, budget, workers=2, stream_workers=2, stream_chunks=6, chunk=0, streaming=False, sel=None):
        """(bounds, streams, largest), or None when a selection group does not fit one chunk"""
        mode = group = None
        if sel is not None:
            mode = (C.c_int * npencil)(*[s[0] for s in sel])
            group = (C.c_int * npencil)(*[s[1] for s in sel])
        bounds = (C.c_int * (npencil + 1))()
        streams, largest = C.c_int(), C.c_int()
        nch = lib.emul_plan(npencil, n, budget, workers, stream_workers, stream_chunks, chunk, int(streaming), mode,
                            group, bounds, C.byref(streams), C.byref(largest))
        if nch < 0:
            return None
        return list(bounds[:nch + 1]), streams.value, largest.value

    return run


def fill_pencils(n):
    """pencils of one full wave of 128-thread blocks on 148 SMs (4 blocks each)"""
    blocks = (n + 127) // 128
    return max(1, (148 * 4 + blocks - 1) // blocks)


def cap_of(npencil, n, budget, workers, stream_workers, streaming):
    """pencils one chunk stream's workspace holds"""
    w = max(1, min(stream_workers if streaming else workers, npencil // fill_pencils(n)))
    return max(1, min(budget // w, 1024))


GOLDEN = [
    # name, (npencil, n, budget, workers, stream_workers, stream_chunks, chunk, streaming, sel), (bounds, streams, largest)
    ("cfg2_resident", (408, 1000, BIG, 2, 2, 6, 0, False, None), ([0, 204, 408], 2, 204)),
    ("cfg2_streamed", (408, 1000, BIG, 2, 2, 6, 0, True, None), ([0, 99, 185, 260, 321, 371, 408], 2, 99)),
    ("chunk37_resident", (408, 1000, BIG, 2, 2, 6, 37, False, None),
     ([0, 37, 74, 111, 148, 185, 222, 259, 296, 333, 370, 407, 408], 2, 37)),
    ("chunk37_streamed", (408, 1000, BIG, 2, 2, 6, 37, True, None),
     ([0, 37, 74, 111, 148, 185, 222, 259, 296, 333, 370, 407, 408], 2, 37)),
    ("stream_workers1", (408, 1000, BIG, 2, 1, 6, 0, True, None), ([0, 99, 185, 260, 321, 371, 408], 1, 99)),
    ("stream_chunks3", (408, 1000, BIG, 2, 2, 3, 0, True, None), ([0, 136, 272, 408], 2, 136)),
    ("budget150_resident", (408, 1000, 150, 2, 2, 6, 0, False, None), ([0, 68, 136, 204, 272, 340, 408], 2, 68)),
    ("budget150_streamed", (408, 1000, 150, 2, 2, 6, 0, True, None), ([0, 99, 185, 260, 321, 371, 408], 2, 99)),
    ("budget100_streamed", (408, 1000, 100, 2, 2, 6, 0, True, None),
     ([0, 46, 92, 138, 184, 230, 276, 322, 368, 408], 2, 46)),
    ("cfg2_select_resident", (408, 1000, BIG, 2, 2, 6, 0, False, SEL51), ([0, 204, 408], 2, 204)),
    ("cfg2_select_streamed", (408, 1000, BIG, 2, 2, 6, 0, True, SEL51), ([0, 204, 408], 2, 204)),
    ("select_groups_of_30", (408, 1000, BIG, 2, 2, 6, 0, False, SEL30), ([0, 210, 408], 2, 210)),
    ("select_group_over_cap", (408, 1000, 60, 2, 2, 6, 0, True, SEL51), None),
    ("select_group_over_cap_forced_chunk", (408, 1000, 60, 2, 2, 6, 20, True, SEL51),
     ([0, 51, 102, 153, 204, 255, 306, 357, 408], 2, 51)),
    ("cfg4_resident", (21, 4000, BIG, 2, 2, 6, 0, False, None), ([0, 21], 1, 21)),
    ("cfg4_streamed", (21, 4000, BIG, 2, 2, 6, 0, True, None), ([0, 11, 21], 1, 11)),
    ("one_pencil", (1, 1000, BIG, 2, 2, 6, 0, True, None), ([0, 1], 1, 1)),
    ("two_pencils", (2, 1000, BIG, 2, 2, 6, 0, True, None), ([0, 2], 1, 2)),
    ("three_pencils", (3, 1000, BIG, 2, 2, 6, 0, False, None), ([0, 3], 1, 3)),
]


@pytest.mark.parametrize("args,want", [g[1:] for g in GOLDEN], ids=[g[0] for g in GOLDEN])
def test_golden(plan, args, want):
    assert plan(*args) == (None if want is None else want)


def random_selection(rng, npencil):
    sel, gid = [], 0
    while len(sel) < npencil:
        mode = rng.choice([0, 1, 1])
        sel += [(mode, rng.choice([gid, gid, -1]) if mode else -1)] * rng.randint(1, 120)
        gid += 1
    return sel[:npencil]


def group_runs(sel):
    """lengths of the runs of consecutive pencils that share one selection group"""
    runs, i = [], 0
    while i < len(sel):
        j = i
        if sel[i][0] and sel[i][1] >= 0:
            while j + 1 < len(sel) and sel[j + 1][0] and sel[j + 1][1] == sel[i][1]:
                j += 1
        runs.append((i, j + 1))
        i = j + 1
    return runs


def test_invariants_seeded_sweep(plan):
    rng = random.Random(20261022)
    errors = 0
    for _ in range(4000):
        npencil = rng.choice([1, 2, 3, 21, 408, rng.randint(1, 1500)])
        n = rng.choice([100, 1000, 4000, rng.randint(1, 6000)])
        budget = rng.choice([BIG, rng.randint(1, 400)])
        workers, stream_workers, stream_chunks = rng.randint(1, 8), rng.randint(1, 8), rng.randint(1, 12)
        chunk = rng.choice([0, 0, 0, rng.randint(1, 300)])
        streaming = rng.random() < 0.5
        sel = random_selection(rng, npencil) if rng.random() < 0.4 else None
        got = plan(npencil, n, budget, workers, stream_workers, stream_chunks, chunk, streaming, sel)
        cap = cap_of(npencil, n, budget, workers, stream_workers, streaming)
        runs = group_runs(sel) if sel is not None and any(s[0] for s in sel) else []
        if got is None:
            # only a selection batch without a forced chunk size can be refused
            assert runs and chunk == 0
            errors += 1
            continue
        # a selection group larger than one stream's workspace cannot be planned without a forced chunk size
        assert not (chunk == 0 and runs and max(b - a for a, b in runs) > cap)
        bounds, streams, largest = got
        sizes = [b - a for a, b in zip(bounds, bounds[1:])]
        assert bounds[0] == 0 and bounds[-1] == npencil
        assert all(s > 0 for s in sizes)
        assert largest == max(sizes)
        assert 1 <= streams <= len(sizes)
        nch = len(sizes)
        shrinking = chunk == 0 and not runs and streaming and nch >= 4 and cap * (nch + 5) >= 2 * npencil
        if shrinking:
            # weights nch+2 .. 3: sizes do not grow (but for the rounding of a bound, in small batches), and the first
            # chunk is (nch+2)/nch of the cap at most (plus one for the rounding)
            assert all(b <= a + 1 for a, b in zip(sizes, sizes[1:]))
            assert sizes == sorted(sizes, reverse=True) or npencil < 8 * nch
            assert largest * nch <= cap * (nch + 2) + nch
        elif chunk == 0:
            assert largest <= cap
        for a, b in runs:
            assert not any(a < x < b for x in bounds), "a selection group was split"
    assert 0 < errors < 4000
