"""The locate walk of record_scan.cuh (gbwt_locate) run on the CPU over the product's device layout, against the oracle's
document array. The walk must be right for any valid sample set, so the table is built here from the document array: a
random subset of the positions plus every sequence's last node, at several densities. CPU only; tests/hostsim is test
infrastructure, not a fallback."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from locate_oracle import NONE, OCCURRENCE, DocumentArray
from oracle import oracle as orc
from test_oracle_locate import FIXTURES, GOLDEN, random_graph

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SAMPLE = np.dtype([("offset", "<u4"), ("seq", "<u4"), ("index", "<u8")])  # LocateSample (layout.h)
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        tmp = tempfile.mkdtemp(prefix="gbwt_hostsim_locate_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libhostsim_locate.so")
        csrc = os.path.join(ROOT, "gbwt-rs_b200", "csrc")
        subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-fopenmp", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", out,
                        os.path.join(HERE, "hostsim", "hostsim_locate.cpp"), os.path.join(csrc, "layout_builder.cpp"),
                        os.path.join(csrc, "sds_loader.cpp"), "-ldl"], check=True, capture_output=True)
        L = C.CDLL(out)
        p, u64 = C.c_void_p, C.c_uint64
        L.hl_load.restype, L.hl_load.argtypes = p, [p, C.c_size_t, C.c_int, C.c_char_p, C.c_size_t]
        L.hl_free.argtypes = [p]
        L.hl_records.restype, L.hl_records.argtypes = u64, [p]
        L.hl_walk_limit.restype, L.hl_walk_limit.argtypes = u64, [p]
        L.hl_locate.argtypes = [p, p, p, u64, p, C.c_size_t, p, p]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def sample_table(da, keep):
    """(first, samples) of the positions where `keep` is set (slot order = record order, then offset order)."""
    chosen = np.concatenate([[0], np.cumsum(keep)]).astype(np.uint64)
    first = np.ascontiguousarray(chosen[da.first.astype(np.int64)].astype(np.uint32))
    slots = np.flatnonzero(keep)
    samples = np.zeros(len(slots) + 1, SAMPLE)  # (one spare entry: an empty table still has an address)
    offsets = np.arange(len(da.seq), dtype=np.uint64) - np.repeat(da.first[:-1], np.diff(da.first).astype(np.int64))
    samples["offset"][:-1] = offsets[slots]
    samples["seq"][:-1] = da.seq[slots]
    samples["index"][:-1] = da.idx[slots]
    return first, samples


def run_locate(image, layout, da, keep, positions):
    arr = np.frombuffer(image, np.uint8).copy()
    err = C.create_string_buffer(256)
    h = lib().hl_load(_p(arr), arr.nbytes, layout, err, 256)
    assert h, err.value
    try:
        assert lib().hl_records(h) == da.records
        first, samples = sample_table(da, keep)
        positions = np.ascontiguousarray(positions, orc.POS_DTYPE)
        out = np.zeros(len(positions), OCCURRENCE)
        steps = np.zeros(len(positions), np.uint64)
        lib().hl_locate(h, _p(first), _p(samples), lib().hl_walk_limit(h), _p(positions), len(positions), _p(out), _p(steps))
        return out, steps
    finally:
        lib().hl_free(h)


def invalid_positions(g):
    return np.array([(0, 0), (g.first_node() - 1 if g.first_node() else 0, 0), (g.alphabet_size(), 0), (g.alphabet_size() + 5, 1),
                     (g.first_node(), 2**40), (g.first_node(), 2**32)], orc.POS_DTYPE)


def check(image, layout, seed):
    g = orc.GBWT.load(image)
    da = DocumentArray(g)
    assert da.ok
    positions = np.concatenate([da.positions(), invalid_positions(g)])
    want = da.locate_batch(positions)
    lengths = np.bincount(da.seq.astype(np.int64), minlength=g.sequences())
    last = da.idx == lengths[da.seq.astype(np.int64)] - 1
    rng = np.random.default_rng(seed)
    for density in (1.0, 0.5, 0.1, 0.0):
        keep = (rng.random(len(da.seq)) < density) | last
        got, steps = run_locate(image, layout, da, keep, positions)
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), f"density {density}"
        if density == 1.0:
            assert not steps.any()
    # no samples but the last nodes: every walk runs to its sequence's end
    got, steps = run_locate(image, layout, da, last, positions[:len(da.seq)])
    assert np.array_equal(steps, (lengths[da.seq.astype(np.int64)] - 1 - da.idx.astype(np.int64)).astype(np.uint64))


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("name", FIXTURES)
def test_fixtures(name, layout):
    check(open(os.path.join(GOLDEN, name), "rb").read(), layout, 1)


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("bidirectional", [True, False])
@pytest.mark.parametrize("seed", range(6))
def test_random_graphs(seed, bidirectional, layout):
    img, _ = random_graph(seed, bidirectional)
    check(img, layout, seed)


def test_walk_gives_up_without_samples():
    """No sample at all (a damaged table): every walk ends as none, within the bound it is given."""
    img, _ = random_graph(3)
    g = orc.GBWT.load(img)
    da = DocumentArray(g)
    got, _ = run_locate(img, 0, da, np.zeros(len(da.seq), bool), da.positions())
    assert np.all(got["sequence"] == NONE) and np.all(got["index"] == NONE)
