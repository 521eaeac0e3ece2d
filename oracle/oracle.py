"""ctypes binding for the CPU oracle (oracle/gbwt_oracle.c) -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module. The product package (gbwt-rs_b200/) never does.

The wrapper mirrors the reference's API names (gbwt-rs src/gbwt.rs:208-385) so the parity
tests read like the reference's own tests; `None` results come back as Python `None`.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

STATE_DTYPE = np.dtype([("node", "<u8"), ("start", "<u8"), ("end", "<u8")])
BDSTATE_DTYPE = np.dtype([("forward", STATE_DTYPE), ("reverse", STATE_DTYPE)])
POS_DTYPE = np.dtype([("node", "<u8"), ("offset", "<u8")])
RUN_DTYPE = np.dtype([("value", "<u8"), ("len", "<u8")])


class Pos(C.Structure):
    _fields_ = [("node", C.c_uint64), ("offset", C.c_uint64)]


class Run(C.Structure):
    _fields_ = [("value", C.c_uint64), ("len", C.c_uint64)]


class State(C.Structure):
    _fields_ = [("node", C.c_uint64), ("start", C.c_uint64), ("end", C.c_uint64)]


class BDState(C.Structure):
    _fields_ = [("forward", State), ("reverse", State)]


_NATIVE_DIR = None


def build(native: bool = False, force: bool = False) -> str:
    """Compile the oracle with the committed Makefile; returns the .so path. The -march=native copy is built for the host
    that runs it, so it goes to a temporary directory of this process (removed at exit), never into the tree: the
    benchmark uses it and may run from a read-only tree."""
    global _NATIVE_DIR
    if native:
        if _NATIVE_DIR is None:
            _NATIVE_DIR = tempfile.TemporaryDirectory(prefix="gbwt_oracle_")
        path = os.path.join(_NATIVE_DIR.name, "libgbwt_oracle_native.so")
    else:
        path = os.path.join(_HERE, "libgbwt_oracle.so")
    src = [os.path.join(_HERE, f) for f in ("gbwt_oracle.c", "gbwt_oracle.h", "Makefile")]
    stale = (not os.path.exists(path)) or any(os.path.getmtime(s) > os.path.getmtime(path) for s in src)
    if force or stale:
        cmd = ["make", "-C", _HERE, "-B", f"OUT={path}"]
        if native:
            cmd.append("MARCH=native")
        subprocess.run(cmd, check=True, capture_output=True)
    return path


_LIBS = {}


def lib(native: bool = False) -> C.CDLL:
    if native not in _LIBS:
        try:
            path = build(native=native)
        except Exception:
            if not native:
                raise
            path = build(native=False)
        L = C.CDLL(path)
        u64, p = C.c_uint64, C.c_void_p
        L.orc_load_bytes.restype = p
        L.orc_load_bytes.argtypes = [p, C.c_size_t, C.c_char_p, C.c_size_t]
        L.orc_load_file.restype = p
        L.orc_load_file.argtypes = [C.c_char_p, C.c_char_p, C.c_size_t]
        L.orc_from_records.restype = p
        L.orc_from_records.argtypes = [u64, p, p, p, p, u64, u64, u64, u64, C.c_int]
        L.orc_free.argtypes = [p]
        for name in ("len", "sequences", "alphabet_size", "alphabet_offset", "effective_size", "first_node",
                     "flags", "bwt_records", "bwt_data_len"):
            f = getattr(L, "orc_" + name)
            f.restype = u64
            f.argtypes = [p]
        L.orc_bwt_data.restype = p
        L.orc_bwt_data.argtypes = [p]
        L.orc_has_node.argtypes = [p, u64]
        L.orc_is_bidirectional.argtypes = [p]
        L.orc_record_bytes.argtypes = [p, u64, C.POINTER(u64), C.POINTER(u64)]
        L.orc_record_outdegree.restype = C.c_int64
        L.orc_record_outdegree.argtypes = [p, u64]
        L.orc_record_edge.argtypes = [p, u64, u64, C.POINTER(Pos)]
        L.orc_record_len.restype = C.c_int64
        L.orc_record_len.argtypes = [p, u64]
        L.orc_record_lf.argtypes = [p, u64, u64, C.POINTER(Pos)]
        L.orc_record_follow.argtypes = [p, u64, u64, u64, u64, C.POINTER(u64), C.POINTER(u64)]
        L.orc_record_bd_follow.argtypes = [p, u64, u64, u64, u64, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64)]
        L.orc_record_decompress.restype = C.c_int64
        L.orc_record_decompress.argtypes = [p, u64, p, u64]
        L.orc_record_predecessor_at.argtypes = [p, u64, u64, C.POINTER(u64)]
        L.orc_record_offset_to.argtypes = [p, u64, Pos, C.POINTER(u64)]
        L.orc_find.argtypes = [p, u64, C.POINTER(State)]
        L.orc_extend.argtypes = [p, C.POINTER(State), u64, C.POINTER(State)]
        L.orc_bd_find.argtypes = [p, u64, C.POINTER(BDState)]
        L.orc_extend_forward.argtypes = [p, C.POINTER(BDState), u64, C.POINTER(BDState)]
        L.orc_extend_backward.argtypes = [p, C.POINTER(BDState), u64, C.POINTER(BDState)]
        L.orc_start.argtypes = [p, u64, C.POINTER(Pos)]
        L.orc_forward.argtypes = [p, Pos, C.POINTER(Pos)]
        L.orc_backward.argtypes = [p, Pos, C.POINTER(Pos)]
        L.orc_sequence.restype = C.c_int64
        L.orc_sequence.argtypes = [p, u64, p, u64]
        L.orc_find_extend_batch.argtypes = [p, p, u64, u64, p, C.c_int]
        L.orc_find_extend_ragged.argtypes = [p, p, p, u64, p, C.c_int]
        L.orc_find_batch.argtypes = [p, p, u64, p, C.c_int]
        L.orc_extend_batch.argtypes = [p, p, p, u64, p, C.c_int]
        L.orc_bd_find_batch.argtypes = [p, p, u64, p, C.c_int]
        L.orc_bd_extend_batch.argtypes = [p, p, p, u64, C.c_int, p, C.c_int]
        L.orc_bd_search_batch.argtypes = [p, p, p, p, p, p, u64, p, C.c_int]
        L.orc_forward_batch.argtypes = [p, p, u64, p, C.c_int]
        L.orc_sequence_lengths.argtypes = [p, p, u64, p, C.c_int]
        L.orc_extract_batch.argtypes = [p, p, u64, p, p, C.c_int]
        L.orc_follow.restype = C.c_int64
        L.orc_follow.argtypes = [p, C.POINTER(BDState), C.c_int, p, u64]
        L.orc_follow_counts.argtypes = [p, p, u64, C.c_int, p, C.c_int]
        L.orc_follow_batch.argtypes = [p, p, u64, C.c_int, p, p, C.c_int]
        L.orc_has_graph.argtypes = [p]
        L.orc_graph_sequences.restype = u64
        L.orc_graph_sequences.argtypes = [p]
        L.orc_node_sequence.restype = C.c_int64
        L.orc_node_sequence.argtypes = [p, u64, C.POINTER(C.c_void_p)]
        L.orc_reverse_complement.argtypes = [p, u64, p]
        L.orc_extract_dna.restype = C.c_int64
        L.orc_extract_dna.argtypes = [p, u64, C.c_uint8, p, u64]
        L.orc_dna_lengths.argtypes = [p, p, u64, p, C.c_int]
        L.orc_extract_dna_batch.argtypes = [p, p, u64, C.c_uint8, p, p, C.c_int]
        L.orc_find_extend_bytes.restype = u64
        L.orc_find_extend_bytes.argtypes = [p, p, u64, u64, C.c_int]
        L.orc_extract_bytes.restype = u64
        L.orc_extract_bytes.argtypes = [p, p, u64, C.c_int]
        L.orc_bytecode_write.restype = C.c_size_t
        L.orc_bytecode_write.argtypes = [p, u64]
        L.orc_bytecode_next.argtypes = [p, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(u64)]
        L.orc_rle_write.restype = C.c_size_t
        L.orc_rle_write.argtypes = [p, u64, Run]
        L.orc_rle_next.argtypes = [p, C.c_size_t, C.POINTER(C.c_size_t), u64, C.POINTER(Run)]
        _LIBS[native] = L
    return _LIBS[native]


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _u64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint64)


# ---- codecs -------------------------------------------------------------------------------

def bytecode_encode(values: Sequence[int]) -> bytes:
    L = lib()
    buf = C.create_string_buffer(10)
    out = bytearray()
    for v in values:
        n = L.orc_bytecode_write(buf, v)
        out += buf.raw[:n]
    return bytes(out)


def bytecode_decode(data: bytes) -> list:
    L = lib()
    pos = C.c_size_t(0)
    v = C.c_uint64(0)
    out = []
    buf = C.create_string_buffer(bytes(data), len(data))
    while L.orc_bytecode_next(buf, len(data), C.byref(pos), C.byref(v)):
        out.append(v.value)
    return out


def rle_encode(sigma: int, runs: Sequence[tuple]) -> bytes:
    L = lib()
    buf = C.create_string_buffer(24)
    out = bytearray()
    for value, length in runs:
        n = L.orc_rle_write(buf, sigma, Run(value, length))
        out += buf.raw[:n]
    return bytes(out)


def rle_decode(sigma: int, data: bytes) -> list:
    L = lib()
    pos = C.c_size_t(0)
    r = Run()
    out = []
    buf = C.create_string_buffer(bytes(data), len(data))
    while L.orc_rle_next(buf, len(data), C.byref(pos), sigma, C.byref(r)):
        out.append((r.value, r.len))
    return out


# ---- the index ----------------------------------------------------------------------------

def reverse_complement(seq: bytes) -> bytes:
    """support::reverse_complement, src/support.rs:104-110."""
    src = np.frombuffer(bytes(seq), dtype=np.uint8).copy()
    out = np.zeros(len(src), dtype=np.uint8)
    lib().orc_reverse_complement(_ptr(src), len(src), _ptr(out))
    return out.tobytes()


def _state(s: State) -> tuple:
    return (s.node, s.start, s.end)


def _bd(s: BDState) -> tuple:
    return (_state(s.forward), _state(s.reverse))


class GBWT:
    """CPU oracle index. Method names follow gbwt-rs `GBWT` (src/gbwt.rs)."""

    def __init__(self, handle, native: bool = False):
        if not handle:
            raise ValueError("oracle: null handle")
        self._h = C.c_void_p(handle)
        self._L = lib(native)

    @classmethod
    def load(cls, path_or_bytes, native: bool = False) -> "GBWT":
        L = lib(native)
        err = C.create_string_buffer(256)
        if isinstance(path_or_bytes, (bytes, bytearray, memoryview, np.ndarray)):
            arr = np.frombuffer(path_or_bytes, dtype=np.uint8) if not isinstance(path_or_bytes, np.ndarray) else path_or_bytes
            arr = np.ascontiguousarray(arr)
            h = L.orc_load_bytes(_ptr(arr), arr.nbytes, err, 256)
        else:
            h = L.orc_load_file(os.fsencode(path_or_bytes), err, 256)
        if not h:
            raise IOError("InvalidData: " + err.value.decode())
        return cls(h, native)

    @classmethod
    def from_records(cls, edges, runs, sequences=0, size=0, offset=0, alphabet_size=None, bidirectional=False) -> "GBWT":
        """BWTBuilder analogue (src/bwt.rs:211-254): `edges[i]` = [(node, offset)], `runs[i]` = [(value, len)]."""
        L = lib()
        n = len(edges)
        ec = _u64([len(e) for e in edges])
        rc = _u64([len(r) for r in runs])
        ef = np.array([x for e in edges for x in e], dtype=np.uint64).reshape(-1, 2) if ec.sum() else np.zeros((0, 2), np.uint64)
        rf = np.array([x for r in runs for x in r], dtype=np.uint64).reshape(-1, 2) if rc.sum() else np.zeros((0, 2), np.uint64)
        ef = np.ascontiguousarray(ef)
        rf = np.ascontiguousarray(rf)
        if alphabet_size is None:
            alphabet_size = n + offset
        h = L.orc_from_records(n, _ptr(ec), _ptr(ef), _ptr(rc), _ptr(rf), sequences, size, offset, alphabet_size,
                               1 if bidirectional else 0)
        return cls(h)

    def __del__(self):
        try:
            if self._h:
                self._L.orc_free(self._h)
                self._h = None
        except Exception:
            pass

    # statistics (src/gbwt.rs:105-175)
    def len(self): return self._L.orc_len(self._h)
    def sequences(self): return self._L.orc_sequences(self._h)
    def alphabet_size(self): return self._L.orc_alphabet_size(self._h)
    def alphabet_offset(self): return self._L.orc_alphabet_offset(self._h)
    def effective_size(self): return self._L.orc_effective_size(self._h)
    def first_node(self): return self._L.orc_first_node(self._h)
    def has_node(self, i): return bool(self._L.orc_has_node(self._h, i))
    def is_bidirectional(self): return bool(self._L.orc_is_bidirectional(self._h))
    def flags(self): return self._L.orc_flags(self._h)
    def bwt_records(self): return self._L.orc_bwt_records(self._h)

    def bwt_data(self) -> bytes:
        n = self._L.orc_bwt_data_len(self._h)
        return C.string_at(self._L.orc_bwt_data(self._h), n)

    def record_bytes(self, i) -> Optional[tuple]:
        s, e = C.c_uint64(), C.c_uint64()
        if not self._L.orc_record_bytes(self._h, i, C.byref(s), C.byref(e)):
            return None
        return (s.value, e.value)

    def record_starts(self) -> np.ndarray:
        return np.array([self.record_bytes(i)[0] for i in range(self.bwt_records())], dtype=np.uint64)

    # record level (src/bwt.rs:329-657)
    def record_outdegree(self, rec):
        n = self._L.orc_record_outdegree(self._h, rec)
        return None if n < 0 else n

    def record_edges(self, rec):
        n = self.record_outdegree(rec)
        if n is None:
            return None
        out = []
        p = Pos()
        for r in range(n):
            self._L.orc_record_edge(self._h, rec, r, C.byref(p))
            out.append((p.node, p.offset))
        return out

    def record_len(self, rec):
        n = self._L.orc_record_len(self._h, rec)
        return None if n < 0 else n

    def record_lf(self, rec, i):
        p = Pos()
        return (p.node, p.offset) if self._L.orc_record_lf(self._h, rec, i, C.byref(p)) else None

    def record_follow(self, rec, start, end, node):
        s, e = C.c_uint64(), C.c_uint64()
        ok = self._L.orc_record_follow(self._h, rec, start, end, node, C.byref(s), C.byref(e))
        return (s.value, e.value) if ok else None

    def record_bd_follow(self, rec, start, end, node):
        s, e, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        ok = self._L.orc_record_bd_follow(self._h, rec, start, end, node, C.byref(s), C.byref(e), C.byref(c))
        return ((s.value, e.value), c.value) if ok else None

    def record_decompress(self, rec):
        n = self._L.orc_record_decompress(self._h, rec, None, 0)
        if n < 0:
            return None
        out = np.zeros(n, dtype=POS_DTYPE)
        self._L.orc_record_decompress(self._h, rec, _ptr(out), n)
        return [(int(a), int(b)) for a, b in out]

    def record_predecessor_at(self, rec, i):
        v = C.c_uint64()
        return v.value if self._L.orc_record_predecessor_at(self._h, rec, i, C.byref(v)) else None

    def record_offset_to(self, rec, pos):
        v = C.c_uint64()
        return v.value if self._L.orc_record_offset_to(self._h, rec, Pos(*pos), C.byref(v)) else None

    # GBWT level (src/gbwt.rs:208-385); states are (node, start, end) tuples
    def find(self, node):
        s = State()
        return _state(s) if self._L.orc_find(self._h, node, C.byref(s)) else None

    def extend(self, state, node):
        s = State(*state)
        o = State()
        return _state(o) if self._L.orc_extend(self._h, C.byref(s), node, C.byref(o)) else None

    def _bdret(self, rc, o):
        if rc < 0:
            raise AssertionError("Bidirectional search requires a bidirectional GBWT")
        return _bd(o) if rc else None

    def bd_find(self, node):
        o = BDState()
        return self._bdret(self._L.orc_bd_find(self._h, node, C.byref(o)), o)

    def extend_forward(self, state, node):
        s = BDState(State(*state[0]), State(*state[1]))
        o = BDState()
        return self._bdret(self._L.orc_extend_forward(self._h, C.byref(s), node, C.byref(o)), o)

    def extend_backward(self, state, node):
        s = BDState(State(*state[0]), State(*state[1]))
        o = BDState()
        return self._bdret(self._L.orc_extend_backward(self._h, C.byref(s), node, C.byref(o)), o)

    def start(self, seq_id):
        p = Pos()
        return (p.node, p.offset) if self._L.orc_start(self._h, seq_id, C.byref(p)) else None

    def forward(self, pos):
        p = Pos()
        return (p.node, p.offset) if self._L.orc_forward(self._h, Pos(*pos), C.byref(p)) else None

    def backward(self, pos):
        p = Pos()
        rc = self._L.orc_backward(self._h, Pos(*pos), C.byref(p))
        if rc < 0:
            raise AssertionError("Following sequences backward requires a bidirectional GBWT")
        return (p.node, p.offset) if rc else None

    def sequence(self, seq_id):
        n = self._L.orc_sequence(self._h, seq_id, None, 0)
        if n < 0:
            return None
        out = np.zeros(n, dtype=np.uint64)
        self._L.orc_sequence(self._h, seq_id, _ptr(out), n)
        return [int(x) for x in out]

    # batch drivers
    def find_extend_batch(self, patterns: np.ndarray, threads: int = 0) -> np.ndarray:
        patterns = _u64(patterns)
        n, k = patterns.shape
        out = np.zeros(n, dtype=STATE_DTYPE)
        self._L.orc_find_extend_batch(self._h, _ptr(patterns), n, k, _ptr(out), threads)
        return out

    def find_extend_ragged(self, nodes, offsets, threads: int = 0) -> np.ndarray:
        nodes, offsets = _u64(nodes), _u64(offsets)
        n = len(offsets) - 1
        out = np.zeros(n, dtype=STATE_DTYPE)
        self._L.orc_find_extend_ragged(self._h, _ptr(nodes), _ptr(offsets), n, _ptr(out), threads)
        return out

    def find_batch(self, nodes, threads: int = 0) -> np.ndarray:
        nodes = _u64(nodes)
        out = np.zeros(len(nodes), dtype=STATE_DTYPE)
        self._L.orc_find_batch(self._h, _ptr(nodes), len(nodes), _ptr(out), threads)
        return out

    def extend_batch(self, states: np.ndarray, nodes, threads: int = 0) -> np.ndarray:
        states = np.ascontiguousarray(states, dtype=STATE_DTYPE)
        nodes = _u64(nodes)
        out = np.zeros(len(nodes), dtype=STATE_DTYPE)
        self._L.orc_extend_batch(self._h, _ptr(states), _ptr(nodes), len(nodes), _ptr(out), threads)
        return out

    def bd_find_batch(self, nodes, threads: int = 0) -> np.ndarray:
        nodes = _u64(nodes)
        out = np.zeros(len(nodes), dtype=BDSTATE_DTYPE)
        if self._L.orc_bd_find_batch(self._h, _ptr(nodes), len(nodes), _ptr(out), threads) < 0:
            raise AssertionError("Bidirectional search requires a bidirectional GBWT")
        return out

    def bd_extend_batch(self, states: np.ndarray, nodes, backward: bool, threads: int = 0) -> np.ndarray:
        states = np.ascontiguousarray(states, dtype=BDSTATE_DTYPE)
        nodes = _u64(nodes)
        out = np.zeros(len(nodes), dtype=BDSTATE_DTYPE)
        rc = self._L.orc_bd_extend_batch(self._h, _ptr(states), _ptr(nodes), len(nodes), 1 if backward else 0, _ptr(out), threads)
        if rc < 0:
            raise AssertionError("Bidirectional search requires a bidirectional GBWT")
        return out

    def bd_search_batch(self, nodes, offsets, first, start, end, threads: int = 0) -> np.ndarray:
        nodes, offsets, first, start, end = map(_u64, (nodes, offsets, first, start, end))
        n = len(first)
        out = np.zeros(n, dtype=BDSTATE_DTYPE)
        rc = self._L.orc_bd_search_batch(self._h, _ptr(nodes), _ptr(offsets), _ptr(first), _ptr(start), _ptr(end), n, _ptr(out), threads)
        if rc < 0:
            raise AssertionError("Bidirectional search requires a bidirectional GBWT")
        return out

    def follow(self, state, backward: bool = False):
        """GBZ::follow_forward / follow_backward (src/gbz.rs:519-544): list of extensions, or None."""
        s = BDState(State(*state[0]), State(*state[1]))
        n = self._L.orc_follow(self._h, C.byref(s), 1 if backward else 0, None, 0)
        if n < 0:
            return None
        out = np.zeros(n, dtype=BDSTATE_DTYPE)
        self._L.orc_follow(self._h, C.byref(s), 1 if backward else 0, _ptr(out), n)
        return [((int(o["forward"]["node"]), int(o["forward"]["start"]), int(o["forward"]["end"])),
                 (int(o["reverse"]["node"]), int(o["reverse"]["start"]), int(o["reverse"]["end"]))) for o in out]

    def follow_batch(self, states: np.ndarray, backward: bool = False, threads: int = 0):
        """Returns (offsets, extensions, counts); counts[i] = 2^64-1 where the reference returns None."""
        states = np.ascontiguousarray(states, dtype=BDSTATE_DTYPE)
        n = len(states)
        counts = np.zeros(n, dtype=np.uint64)
        self._L.orc_follow_counts(self._h, _ptr(states), n, 1 if backward else 0, _ptr(counts), threads)
        sizes = np.where(counts == np.uint64(2**64 - 1), np.uint64(0), counts)
        offsets = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum(sizes, out=offsets[1:])
        out = np.zeros(int(offsets[-1]), dtype=BDSTATE_DTYPE)
        self._L.orc_follow_batch(self._h, _ptr(states), n, 1 if backward else 0, _ptr(offsets), _ptr(out), threads)
        return offsets, out, counts

    # node sequences / DNA (GBZ files)
    def has_graph(self): return bool(self._L.orc_has_graph(self._h))
    def graph_sequences(self): return self._L.orc_graph_sequences(self._h)

    def node_sequence(self, node_id):
        """GBZ::sequence(node_id), src/gbz.rs:292-298."""
        ptr = C.c_void_p()
        n = self._L.orc_node_sequence(self._h, node_id, C.byref(ptr))
        return None if n < 0 else C.string_at(ptr.value, n)

    def extract_dna(self, seq_id, endmarker=0):
        """extract_sequence of src/bin/gbz-extract.rs:173-189 for GBWT sequence `seq_id`."""
        n = self._L.orc_extract_dna(self._h, seq_id, endmarker, None, 0)
        if n < 0:
            return None
        out = np.zeros(n, dtype=np.uint8)
        self._L.orc_extract_dna(self._h, seq_id, endmarker, _ptr(out), n)
        return out.tobytes()

    def extract_dna_batch(self, ids, endmarker=0, threads: int = 0):
        ids = _u64(ids)
        lengths = np.zeros(len(ids), dtype=np.uint64)
        self._L.orc_dna_lengths(self._h, _ptr(ids), len(ids), _ptr(lengths), threads)
        sizes = np.where(lengths == np.uint64(2**64 - 1), np.uint64(0), lengths)
        offsets = np.zeros(len(ids) + 1, dtype=np.uint64)
        np.cumsum(sizes, out=offsets[1:])
        out = np.zeros(int(offsets[-1]), dtype=np.uint8)
        self._L.orc_extract_dna_batch(self._h, _ptr(ids), len(ids), endmarker, _ptr(offsets), _ptr(out), threads)
        return offsets, out, lengths

    def forward_batch(self, positions: np.ndarray, threads: int = 0) -> np.ndarray:
        positions = np.ascontiguousarray(positions, dtype=POS_DTYPE)
        out = np.zeros(len(positions), dtype=POS_DTYPE)
        self._L.orc_forward_batch(self._h, _ptr(positions), len(positions), _ptr(out), threads)
        return out

    def sequence_lengths(self, ids, threads: int = 0) -> np.ndarray:
        ids = _u64(ids)
        out = np.zeros(len(ids), dtype=np.uint64)
        self._L.orc_sequence_lengths(self._h, _ptr(ids), len(ids), _ptr(out), threads)
        return out

    def find_extend_bytes(self, patterns: np.ndarray, threads: int = 0) -> int:
        """Algorithmic bytes of SURVEY.md 8(d) for these patterns (reference's compressed records)."""
        patterns = _u64(patterns)
        n, k = patterns.shape
        return int(self._L.orc_find_extend_bytes(self._h, _ptr(patterns), n, k, threads))

    def extract_bytes(self, ids, threads: int = 0) -> int:
        ids = _u64(ids)
        return int(self._L.orc_extract_bytes(self._h, _ptr(ids), len(ids), threads))

    def extract_batch(self, ids, threads: int = 0):
        ids = _u64(ids)
        lengths = self.sequence_lengths(ids, threads)
        lengths = np.where(lengths == np.uint64(2**64 - 1), np.uint64(0), lengths)
        offsets = np.zeros(len(ids) + 1, dtype=np.uint64)
        np.cumsum(lengths, out=offsets[1:])
        nodes = np.zeros(int(offsets[-1]), dtype=np.uint64)
        self._L.orc_extract_batch(self._h, _ptr(ids), len(ids), _ptr(offsets), _ptr(nodes), threads)
        return offsets, nodes


def max_threads() -> int:
    return lib().orc_max_threads()
