"""Document array of a GBWT from the CPU oracle (tests/locate_oracle/da_oracle.c) -- TEST INFRASTRUCTURE ONLY.

`DocumentArray(g)` walks every sequence of the oracle GBWT `g` with GBWT::start / GBWT::forward and records, for every
BWT position, the sequence it lies on and its index there: the answer locate must give, independent of any sampling.
The helper library is compiled into a temporary directory of the process (the benchmark may run from a read-only tree)
and linked against the oracle library that `g` was loaded from.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import oracle as orc  # noqa: E402

OCCURRENCE = np.dtype([("sequence", "<u8"), ("index", "<u8")])
NONE = np.uint64(2**64 - 1)
_LIBS = {}


def _lib(oracle_path: str) -> C.CDLL:
    if oracle_path not in _LIBS:
        tmp = tempfile.mkdtemp(prefix="gbwt_da_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libda_oracle.so")
        subprocess.run(["/usr/bin/gcc", "-O2", "-fPIC", "-shared", "-std=gnu11", "-o", out,
                        os.path.join(HERE, "locate_oracle", "da_oracle.c"), oracle_path], check=True, capture_output=True)
        L = C.CDLL(out)
        p = C.c_void_p
        L.da_layout.restype, L.da_layout.argtypes = C.c_uint64, [p, p]
        L.da_build.restype, L.da_build.argtypes = C.c_int, [p, p, p, p]
        _LIBS[oracle_path] = L
    return _LIBS[oracle_path]


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class DocumentArray:
    """first[r] = slot of record r's first position; seq / idx per slot (UINT64_MAX where no sequence visits it)."""

    def __init__(self, g: "orc.GBWT"):
        L = _lib(g._L._name)  # (the oracle library g was loaded from)
        self.offset, self.first_node = g.alphabet_offset(), g.first_node()
        self.records = g._L.orc_bwt_records(g._h)
        self.first = np.zeros(self.records + 1, np.uint64)
        slots = L.da_layout(g._h, _p(self.first))
        self.seq = np.zeros(slots, np.uint64)
        self.idx = np.zeros(slots, np.uint64)
        self.ok = L.da_build(g._h, _p(self.first), _p(self.seq), _p(self.idx)) == 0

    def document_array(self):
        """(first, occurrences): the occurrence of every position, by record and offset."""
        occ = np.zeros(len(self.seq), OCCURRENCE)
        occ["sequence"], occ["index"] = self.seq, self.idx
        return self.first, occ

    def positions(self):
        """Every (node, offset) of the array, in slot order (POS dtype of the oracle)."""
        lens = np.diff(self.first)
        rec = np.repeat(np.arange(self.records, dtype=np.uint64), lens.astype(np.int64))
        out = np.zeros(len(self.seq), orc.POS_DTYPE)
        out["node"] = rec + np.uint64(self.offset)
        out["offset"] = np.arange(len(self.seq), dtype=np.uint64) - np.repeat(self.first[:-1], lens.astype(np.int64))
        return out

    def locate_batch(self, positions) -> np.ndarray:
        """locate for many positions: (sequence, index), UINT64_MAX in both where there is no such position."""
        positions = np.ascontiguousarray(positions, orc.POS_DTYPE)
        node, off = positions["node"], positions["offset"]
        out = np.full(len(positions), NONE, dtype=np.uint64)
        res = np.zeros(len(positions), OCCURRENCE)
        res["sequence"], res["index"] = out, out
        rec = node - np.uint64(self.offset)
        valid = (node >= np.uint64(self.first_node)) & (rec < np.uint64(self.records))
        r = np.where(valid, rec, 0).astype(np.int64)
        lens = self.first[r + 1] - self.first[r]
        valid &= off < lens
        k = (self.first[r] + np.where(valid, off, 0)).astype(np.int64)
        res["sequence"][valid] = self.seq[k[valid]]
        res["index"][valid] = self.idx[k[valid]]
        return res

    def locate_states(self, states):
        """(offsets, occurrences) of search states, in offset order."""
        states = np.ascontiguousarray(states, orc.STATE_DTYPE)
        sizes = np.where(states["end"] > states["start"], states["end"] - states["start"], np.uint64(0)).astype(np.uint64)
        offsets = np.zeros(len(states) + 1, np.uint64)
        np.cumsum(sizes, out=offsets[1:])
        pos = np.zeros(int(offsets[-1]), orc.POS_DTYPE)
        owner = np.repeat(np.arange(len(states)), sizes.astype(np.int64))
        pos["node"] = states["node"][owner]
        pos["offset"] = states["start"][owner] + (np.arange(len(pos), dtype=np.uint64) - offsets[:-1][owner])
        return offsets, self.locate_batch(pos)


def _mix64(x: np.ndarray) -> np.ndarray:
    """synth/gbwt_synth.c mix64 (splitmix64 finaliser) on uint64 arrays."""
    x = x + np.uint64(0x9E3779B97F4A7C15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def pattern_origins(sites: int, haplotypes: int, n: int, k: int = 32, seed_q: int = 7, q0: int = 0):
    """Where synth.patterns took pattern q from: sequence 2h + o, nodes t .. t + k - 1 (synth_patterns_v). The state a
    find/extend of the pattern reaches must therefore contain the occurrence (2h + o, t + k - 1)."""
    q = np.arange(q0, q0 + n, dtype=np.uint64)
    base = np.uint64(seed_q) + np.uint64(3) * q
    h = _mix64(base) % np.uint64(haplotypes)
    o = _mix64(base + np.uint64(1)) & np.uint64(1)
    t = _mix64(base + np.uint64(2)) % np.uint64(2 * sites + 1 - (k - 1))
    return np.uint64(2) * h + o, t + np.uint64(k - 1)


def states_contain(offsets, occurrences, seqs, idxs) -> bool:
    """Whether the occurrences of state q (occurrences[offsets[q]:offsets[q + 1]]) include (seqs[q], idxs[q]), for every q."""
    n = len(seqs)
    sizes = np.diff(offsets).astype(np.int64)
    owner = np.repeat(np.arange(n), sizes)
    hit = (occurrences["sequence"] == seqs[owner]) & (occurrences["index"] == idxs[owner])
    return bool(np.all(np.bincount(owner[hit], minlength=n) == 1))
