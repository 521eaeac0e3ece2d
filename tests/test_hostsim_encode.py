"""The record encoder shared by the host writer and the device builder (gbwt-rs_b200/csrc/record_encode.h), compiled for
the CPU and compared with tests/gbwt_builder.encode_record over random edge and run lists, outdegrees 1 to 300. CPU only."""
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

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        tmp = tempfile.mkdtemp(prefix="gbwt_hostsim_encode_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libhostsim_encode.so")
        subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-o", out,
                        os.path.join(HERE, "hostsim", "hostsim_encode.cpp")], check=True, capture_output=True)
        L = C.CDLL(out)
        p, u64 = C.c_void_p, C.c_uint64
        L.he_encode_record.restype = u64
        L.he_encode_record.argtypes = [p, u64, p, u64, p]
        _LIB = L
    return _LIB


def encode(edges, runs) -> bytes:
    e = np.array(edges, dtype=np.uint64).reshape(-1, 2)
    r = np.array(runs, dtype=np.uint64).reshape(-1, 2)
    ep, rp = e.ctypes.data_as(C.c_void_p), r.ctypes.data_as(C.c_void_p)
    n = lib().he_encode_record(ep, len(e), rp, len(r), None)
    out = np.zeros(max(n, 1), dtype=np.uint8)
    assert lib().he_encode_record(ep, len(e), rp, len(r), out.ctypes.data_as(C.c_void_p)) == n
    return out[:n].tobytes()


def random_record(rng, sigma):
    nodes = sorted(rng.sample(range(0, 1 << 33), sigma))
    edges = [(v, rng.choice([0, rng.randrange(1 << 7), rng.randrange(1 << 40)])) for v in nodes]
    runs, prev = [], None
    for _ in range(rng.randrange(1, 40)):
        value = rng.randrange(sigma)
        if value == prev and sigma > 1:
            value = (value + 1) % sigma
        threshold = max(1, 256 // sigma)
        length = rng.choice([1, 2, threshold - 1 if threshold > 1 else 1, threshold, threshold + 1, rng.randrange(1, 1 << 20)])
        runs.append((value, length))
        prev = value
    return edges, runs


@pytest.mark.parametrize("sigma", list(range(1, 20)) + [63, 64, 85, 86, 127, 128, 129, 254, 255, 256, 300])
def test_encoder_matches_builder(sigma):
    rng = random.Random(sigma)
    for _ in range(20):
        edges, runs = random_record(rng, sigma)
        assert encode(edges, runs) == gb.encode_record(edges, runs)


def test_every_outdegree_up_to_300():
    rng = random.Random(7)
    for sigma in range(1, 301):
        edges, runs = random_record(rng, sigma)
        assert encode(edges, runs) == gb.encode_record(edges, runs)


def test_empty_record_is_one_zero_byte():
    assert encode([], []) == gb.encode_record([], []) == b"\x00"
