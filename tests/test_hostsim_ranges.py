"""The seek walk of record_scan.cuh (gbwt_seek) run on the CPU over the product's device layout, against the oracle's start +
forward. The walk must be right for any table the checkpoint build can leave, so the tables are made here the way that walk
makes them: slot k of a sequence holds the first flush at or after node k 2^shift, flushes lie at most 32 nodes apart (at
most 2^shift for the small intervals used on the small fixtures), and a sequence that ends before that flush has no slot k.
CPU only; tests/hostsim is test infrastructure, not a fallback."""
import atexit
import ctypes as C
import os
import random
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import gbwt_builder as gb
from oracle import oracle as orc
from test_oracle_locate import FIXTURES, GOLDEN, image_of, random_graph

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CHECKPOINT = np.dtype([("node", "<u4"), ("offset", "<u4"), ("index", "<u8")])  # Checkpoint (layout.h)
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        tmp = tempfile.mkdtemp(prefix="gbwt_hostsim_ranges_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libhostsim_ranges.so")
        csrc = os.path.join(ROOT, "gbwt-rs_b200", "csrc")
        subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-fopenmp", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", out,
                        os.path.join(HERE, "hostsim", "hostsim_ranges.cpp"), os.path.join(csrc, "layout_builder.cpp"),
                        os.path.join(csrc, "sds_loader.cpp"), "-ldl"], check=True, capture_output=True)
        L = C.CDLL(out)
        p = C.c_void_p
        L.hr_load.restype, L.hr_load.argtypes = p, [p, C.c_size_t, C.c_int, C.c_char_p, C.c_size_t]
        L.hr_free.argtypes = [p]
        L.hr_seek.argtypes = [p, p, p, p, C.c_uint32, p, p, C.c_size_t, p, p]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def paths_of(g):
    """Every sequence as its list of positions, by the oracle's start + forward."""
    out = []
    for s in range(g.sequences()):
        pos, p = [], g.start(s)
        while p is not None:
            pos.append(p)
            p = g.forward(p)
        out.append(pos)
    return out


def checkpoint_table(paths, shift, rng):
    """(table, first, seq_len) as k_build_checkpoints leaves them, with flushes at random gaps of at most 32 nodes (at most
    2^shift below 2^6)."""
    interval = 1 << shift
    gap_lo, gap_hi = (31, 32) if interval >= 64 else (1, interval)
    rows, first = [], [0]
    for pos in paths:
        flushes, f = [0], 0
        while f < len(pos):
            f += rng.randint(gap_lo, gap_hi)
            flushes.append(f)
        for k in range(len(pos)):
            at = next((x for x in flushes if x >= k * interval), len(pos))
            if at >= len(pos):
                break
            rows.append((pos[at][0], pos[at][1], at))
        first.append(len(rows))
    table = np.zeros(len(rows) + 1, CHECKPOINT)  # (one spare entry: an empty table still has an address)
    for n, r in enumerate(rows):
        table[n] = r
    return table, np.array(first, np.uint32), np.array([len(p) for p in paths], np.uint64)


def run_seek(image, layout, table, ids, indexes):
    arr = np.frombuffer(image, np.uint8).copy()
    err = C.create_string_buffer(256)
    h = lib().hr_load(_p(arr), arr.nbytes, layout, err, 256)
    assert h, err.value
    try:
        ids, indexes = np.ascontiguousarray(ids, np.uint64), np.ascontiguousarray(indexes, np.uint64)
        out = np.zeros(len(ids), orc.POS_DTYPE)
        steps = np.zeros(len(ids), np.uint64)
        tab, first, seq_len, shift = table if table is not None else (None, None, None, 0)
        lib().hr_seek(h, _p(tab), _p(first), _p(seq_len), shift, _p(ids), _p(indexes), len(ids), _p(out), _p(steps))
        return out, steps
    finally:
        lib().hr_free(h)


def queries(paths, table):
    """Every (s, j), j = len and j = len + 1, s = sequences(), and j at and around every checkpoint index."""
    ids, idx = [], []
    for s, pos in enumerate(paths):
        for j in range(len(pos) + 2):
            ids.append(s); idx.append(j)
    n = len(paths)
    ids += [n, n + 1, 2**64 - 1, 0]
    idx += [0, 0, 0, 2**64 - 1]
    if table is not None:
        tab, first, _, _ = table
        for s in range(n):
            for k in range(int(first[s]), int(first[s + 1])):
                at = int(tab[k]["index"])
                for j in (at - 1, at, at + 1):
                    if j >= 0:
                        ids.append(s); idx.append(j)
    return np.array(ids, np.uint64), np.array(idx, np.uint64)


def expected(paths, ids, idx):
    want = np.zeros(len(ids), orc.POS_DTYPE)
    for q, (s, j) in enumerate(zip(ids.tolist(), idx.tolist())):
        if s < len(paths) and j < len(paths[s]):
            want[q] = paths[s][j]
    return want


def check(image, layout, seed, shifts):
    g = orc.GBWT.load(image)
    paths = paths_of(g)
    rng = random.Random(seed)
    for shift in shifts:
        table = None if shift is None else checkpoint_table(paths, shift, rng) + (shift,)
        ids, idx = queries(paths, table)
        got, steps = run_seek(image, layout, table, ids, idx)
        assert np.array_equal(got.view(np.uint64), expected(paths, ids, idx).view(np.uint64)), f"shift {shift}"
        ok = got["node"] != 0
        if table is not None:
            # a walk never takes more than one interval plus the flush slack
            assert int(steps[ok].max(initial=0)) < (1 << shift) + 32
        else:
            assert np.array_equal(steps[ok], idx[ok])


# None = no checkpoints (walks from start); 40 = slot 0 only
SHIFTS = (None, 0, 1, 2, 3, 6, 40)


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("name", FIXTURES)
def test_fixtures(name, layout):
    check(open(os.path.join(GOLDEN, name), "rb").read(), layout, 1, SHIFTS)


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("bidirectional", [True, False])
@pytest.mark.parametrize("seed", range(6))
def test_random_graphs(seed, bidirectional, layout):
    img, _ = random_graph(seed, bidirectional)
    check(img, layout, seed, SHIFTS)


@pytest.mark.parametrize("seed", range(3))
def test_long_paths(seed):
    """Paths of hundreds of nodes, so that the real interval (2^6 and up, flushes 31 or 32 nodes apart) has many slots."""
    rng = random.Random(seed)
    paths = [[2 * rng.randint(1, 12) + (1 if rng.random() < 0.1 else 0) for _ in range(rng.randint(0, 700))] for _ in range(6)]
    img = image_of(gb.build_bwt(gb.bidirectional_sequences(paths)), True)
    check(img, 0, seed, (None, 6, 7, 8, 40))
