"""gbwt-rs_b200: B200-native batched GBWT search and LF traversal (host-side mirror of the gbwt-rs API).

The package directory is `gbwt-rs_b200/`; import it as `gbwt_rs_b200` (the repo root ships a tiny alias
module, because a hyphen cannot appear in a Python module name).

`GBWT` keeps the method names and result semantics of the reference crate's `GBWT` (gbwt-rs src/gbwt.rs):
`find`, `extend`, `bd_find`, `extend_forward`, `extend_backward`, `start`, `forward`, `backward`, `sequence`
and the statistics accessors. Every method accepts either the reference's scalar arguments (a batch of one,
returning `SearchState` / `BidirectionalState` / `Pos` or `None`) or numpy arrays (a batch, returning
structured arrays in the C ABI's layout). All of them run CUDA kernels through the C ABI of
include/gbwt_b200.h; there is no CPU fallback and importing fails loudly if the library is missing.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Iterator, Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIBRARY = os.environ.get("GBWT_B200_LIBRARY") or os.path.join(_HERE, "libgbwt_b200.so")  # override: development builds

ENDMARKER = 0  # gbwt-rs src/lib.rs:59

STATE_DTYPE = np.dtype([("node", "<u8"), ("start", "<u8"), ("end", "<u8")])
BDSTATE_DTYPE = np.dtype([("forward", STATE_DTYPE), ("reverse", STATE_DTYPE)])
POS_DTYPE = np.dtype([("node", "<u8"), ("offset", "<u8")])
OCCURRENCE_DTYPE = np.dtype([("sequence", "<u8"), ("index", "<u8")])  # gbwt_b200_occurrence

LAYOUT_AUTO, LAYOUT_RUNS = 0, 1
LAYOUT_CHECKPOINTS, LAYOUT_NO_CHECKPOINTS = 0x100, 0x200
LAYOUT_LOCATE = 0x400  # locate samples (GBWT.locate); the `locate=True` keyword of load / from_bytes / from_parts
_LAYOUTS = {"auto": LAYOUT_AUTO, "runs": LAYOUT_RUNS, 0: LAYOUT_AUTO, 1: LAYOUT_RUNS}


def _policy(layout, checkpoints, locate=False) -> int:
    """Layout policy word of the C ABI: body layout + the checkpoint flag (None = the library's default by size) + the
    locate-sample flag."""
    flag = 0 if checkpoints is None else (LAYOUT_CHECKPOINTS if checkpoints else LAYOUT_NO_CHECKPOINTS)
    return _LAYOUTS[layout] | flag | (LAYOUT_LOCATE if locate else 0)

OK, E_INVALID_DATA, E_IO, E_RANGE, E_NOT_BIDIRECTIONAL, E_CUDA, E_ARGUMENT, E_NO_DEVICE = range(8)
E_NO_GRAPH, E_NO_SAMPLES = 8, 9
_U64MAX = np.uint64(2**64 - 1)


class GBWTError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"gbwt_b200 error {code}: {message}")
        self.code = code


def _load_library() -> C.CDLL:
    if not os.path.exists(LIBRARY):
        try:
            from . import build as _build
            _build.build()
        except Exception as exc:  # no silent fallback: the CUDA library is the product
            raise ImportError(f"{LIBRARY} is missing and could not be built ({exc}); run python gbwt-rs_b200/build.py") from exc
    L = C.CDLL(LIBRARY)
    p, u64, sz, i = C.c_void_p, C.c_uint64, C.c_size_t, C.c_int
    pp = C.POINTER(C.c_void_p)
    sig = {
        "gbwt_b200_index_load_file": (i, [C.c_char_p, i, i, pp]),
        "gbwt_b200_index_from_bytes": (i, [p, sz, i, i, pp]),
        "gbwt_b200_index_from_parts": (i, [u64, u64, u64, u64, u64, p, u64, p, u64, i, i, pp]),
        "gbwt_b200_index_destroy": (None, [p]),
        "gbwt_b200_index_serialize": (i, [p, pp, C.POINTER(sz)]),
        "gbwt_b200_index_save_file": (i, [p, C.c_char_p]),
        "gbwt_b200_index_serialize_gbz": (i, [p, pp, C.POINTER(sz)]),
        "gbwt_b200_index_save_gbz_file": (i, [p, C.c_char_p]),
        "gbwt_b200_index_export_ipc": (i, [p, pp, C.POINTER(sz)]),
        "gbwt_b200_index_import_ipc": (i, [p, sz, i, pp]),
        "gbwt_b200_free": (None, [p]),
        "gbwt_b200_last_error": (C.c_char_p, []),
        "gbwt_b200_len": (u64, [p]), "gbwt_b200_sequences": (u64, [p]), "gbwt_b200_alphabet_size": (u64, [p]),
        "gbwt_b200_alphabet_offset": (u64, [p]), "gbwt_b200_effective_size": (u64, [p]), "gbwt_b200_first_node": (u64, [p]),
        "gbwt_b200_has_node": (i, [p, u64]), "gbwt_b200_is_bidirectional": (i, [p]), "gbwt_b200_device": (i, [p]),
        "gbwt_b200_device_bytes": (u64, [p, p]),
        "gbwt_b200_window_info": (None, [p, p]),
        "gbwt_b200_checkpoint_info": (None, [p, p]),
        "gbwt_b200_locate_info": (None, [p, p]),
        "gbwt_b200_locate": (i, [p, p, sz, p]),
        "gbwt_b200_locate_states": (i, [p, p, sz, p, p, p]),
        "gbwt_b200_locate_device": (i, [p, p, sz, p, p]),
        "gbwt_b200_locate_states_device": (i, [p, p, sz, p, p, p, p]),
        "gbwt_b200_find": (i, [p, p, sz, p]),
        "gbwt_b200_extend": (i, [p, p, p, sz, p]),
        "gbwt_b200_find_extend": (i, [p, p, sz, sz, p]),
        "gbwt_b200_find_extend_u32": (i, [p, p, sz, sz, p]),
        "gbwt_b200_find_extend_ragged": (i, [p, p, p, sz, p]),
        "gbwt_b200_bd_find": (i, [p, p, sz, p]),
        "gbwt_b200_extend_forward": (i, [p, p, p, sz, p]),
        "gbwt_b200_extend_backward": (i, [p, p, p, sz, p]),
        "gbwt_b200_bd_search": (i, [p, p, p, p, p, p, sz, p]),
        "gbwt_b200_follow": (i, [p, p, sz, i, p, p, p]),
        "gbwt_b200_follow_device": (i, [p, p, sz, i, p, p, p, p]),
        "gbwt_b200_start": (i, [p, p, sz, p]),
        "gbwt_b200_forward": (i, [p, p, sz, p]),
        "gbwt_b200_backward": (i, [p, p, sz, p]),
        "gbwt_b200_sequence_lengths": (i, [p, p, sz, p]),
        "gbwt_b200_extract": (i, [p, p, sz, p, p, p]),
        "gbwt_b200_find_extend_device": (i, [p, p, sz, sz, p, p]),
        "gbwt_b200_find_extend_u32_device": (i, [p, p, sz, sz, p, p]),
        "gbwt_b200_find_extend_ragged_device": (i, [p, p, p, sz, p, p]),
        "gbwt_b200_find_device": (i, [p, p, sz, p, p]),
        "gbwt_b200_extend_device": (i, [p, p, p, sz, p, p]),
        "gbwt_b200_bd_find_device": (i, [p, p, sz, p, p]),
        "gbwt_b200_bd_extend_device": (i, [p, p, p, sz, i, p, p]),
        "gbwt_b200_bd_search_device": (i, [p, p, p, p, p, p, sz, p, p]),
        "gbwt_b200_forward_device": (i, [p, p, sz, p, p]),
        "gbwt_b200_sequence_lengths_device": (i, [p, p, sz, p, p]),
        "gbwt_b200_extract_device": (i, [p, p, sz, p, p, p, p]),
        "gbwt_b200_index_attach_graph": (i, [p, u64, p, p]),
        "gbwt_b200_has_graph": (i, [p]), "gbwt_b200_graph_sequences": (u64, [p]), "gbwt_b200_graph_bytes": (u64, [p]), "gbwt_b200_skip_bytes": (u64, [p]), "gbwt_b200_run_checkpoint_records": (u64, [p]), "gbwt_b200_dense4_records": (u64, [p]),
        "gbwt_b200_node_sequence_lengths": (i, [p, p, sz, p]),
        "gbwt_b200_node_sequences": (i, [p, p, sz, p, p, p]),
        "gbwt_b200_dna_lengths": (i, [p, p, sz, p]),
        "gbwt_b200_extract_dna": (i, [p, p, sz, C.c_uint8, p, p, p]),
        "gbwt_b200_dna_lengths_device": (i, [p, p, sz, p, p]),
        "gbwt_b200_extract_dna_device": (i, [p, p, sz, C.c_uint8, p, p, p, p]),
        "gbwt_b200_seek": (i, [p, p, p, sz, p]),
        "gbwt_b200_extract_ranges": (i, [p, p, p, p, sz, p, p, p]),
        "gbwt_b200_extract_dna_ranges": (i, [p, p, p, p, sz, p, p, p]),
        "gbwt_b200_seek_device": (i, [p, p, p, sz, p, p]),
        "gbwt_b200_extract_ranges_device": (i, [p, p, p, p, sz, p, p, p, p]),
        "gbwt_b200_extract_dna_ranges_device": (i, [p, p, p, p, sz, p, p, p, p]),
        "gbwt_b200_build_image": (i, [p, p, sz, i, i, pp, C.POINTER(sz), p]),
        "gbwt_b200_build_image_device": (i, [p, p, sz, i, i, p, pp, C.POINTER(sz), p]),
        "gbwt_b200_host_alloc": (p, [sz]), "gbwt_b200_host_free": (None, [p]),
        "gbwt_b200_kernel_launches": (u64, []), "gbwt_b200_version": (C.c_char_p, []),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)  # AttributeError if the library does not export what include/gbwt_b200.h declares
        f.restype, f.argtypes = res, args
    return L


_lib = _load_library()
EXPORTS = None  # filled lazily by exported_symbols()


def library() -> C.CDLL:
    return _lib


def kernel_launches() -> int:
    return int(_lib.gbwt_b200_kernel_launches())


def version() -> str:
    return _lib.gbwt_b200_version().decode()


# ---- value types of the reference API --------------------------------------------------------------

@dataclass(frozen=True)
class Pos:
    """gbwt-rs `Pos` (src/bwt.rs:63-69)."""
    node: int
    offset: int


@dataclass(frozen=True)
class SearchState:
    """gbwt-rs `SearchState` (src/gbwt.rs:454-474): `range` is a Python range like Rust's Range<usize>."""
    node: int
    range: range

    def len(self) -> int:
        return len(self.range)

    def is_empty(self) -> bool:
        return len(self.range) == 0

    def __len__(self) -> int:
        return len(self.range)


@dataclass(frozen=True)
class BidirectionalState:
    """gbwt-rs `BidirectionalState` (src/gbwt.rs:484-528)."""
    forward: SearchState
    reverse: SearchState

    def len(self) -> int:
        return self.forward.len()

    def is_empty(self) -> bool:
        return self.forward.is_empty()

    def flip(self) -> "BidirectionalState":
        return BidirectionalState(self.reverse, self.forward)

    def from_(self):
        """(node id, is_reverse) of the first node on the path (src/gbwt.rs:517-519)."""
        n = self.reverse.node ^ 1
        return (n // 2, bool(n & 1))

    def to(self):
        n = self.forward.node
        return (n // 2, bool(n & 1))


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _u64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint64)


def _is_scalar(x) -> bool:
    return isinstance(x, (int, np.integer))


def _state_rec(s: SearchState):
    return (s.node, s.range.start, s.range.stop)


def _state_obj(rec) -> Optional[SearchState]:
    if int(rec["end"]) <= int(rec["start"]):
        return None
    return SearchState(int(rec["node"]), range(int(rec["start"]), int(rec["end"])))


def _bd_obj(rec) -> Optional[BidirectionalState]:
    f, r = _state_obj(rec["forward"]), _state_obj(rec["reverse"])
    if f is None:
        return None
    return BidirectionalState(f, r)


class GBWT:
    """Device-resident GBWT index. Mirrors gbwt-rs `GBWT` (src/gbwt.rs:95-385)."""

    name = "b200"

    def __init__(self, handle: int):
        self._h = C.c_void_p(handle)

    # -- construction (GBWT::load / serialize::load_from, src/gbwt.rs:402-438) --
    @staticmethod
    def _check(rc: int):
        if rc != OK:
            msg = _lib.gbwt_b200_last_error().decode()
            if rc in (E_INVALID_DATA, E_IO):
                raise IOError(f"InvalidData: {msg}" if rc == E_INVALID_DATA else msg)
            if rc == E_NOT_BIDIRECTIONAL:
                raise AssertionError(msg)  # the reference panics (assert!, src/gbwt.rs:237, 312, 340)
            raise GBWTError(rc, msg)

    @classmethod
    def load(cls, path, device: int = 0, layout="auto", checkpoints=None, locate=False) -> "GBWT":
        h = C.c_void_p()
        cls._check(_lib.gbwt_b200_index_load_file(os.fsencode(path), device, _policy(layout, checkpoints, locate), C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_bytes(cls, image, device: int = 0, layout="auto", checkpoints=None, locate=False) -> "GBWT":
        arr = image if isinstance(image, np.ndarray) else np.frombuffer(image, dtype=np.uint8)
        arr = np.ascontiguousarray(arr)
        h = C.c_void_p()
        cls._check(_lib.gbwt_b200_index_from_bytes(_ptr(arr), arr.nbytes, device, _policy(layout, checkpoints, locate), C.byref(h)))
        return cls(h.value)

    @classmethod
    def build(cls, paths, bidirectional: bool = True, device: int = 0, layout="auto", checkpoints=None, locate=False) -> "GBWT":
        """The GBWT of the given paths, built on the device (build_image), loaded like from_bytes."""
        return cls.from_bytes(build_image(paths, bidirectional, device), device, layout, checkpoints, locate)

    @classmethod
    def from_parts(cls, sequences, size, offset, alphabet_size, flags, bwt_bytes, record_starts, device: int = 0,
                   layout="auto", locate=False) -> "GBWT":
        data = np.ascontiguousarray(np.frombuffer(bytes(bwt_bytes), dtype=np.uint8))
        starts = _u64(record_starts)
        h = C.c_void_p()
        cls._check(_lib.gbwt_b200_index_from_parts(sequences, size, offset, alphabet_size, flags, _ptr(data), data.nbytes,
                                                   _ptr(starts), len(starts), device, _policy(layout, None, locate), C.byref(h)))
        return cls(h.value)

    def attach_graph(self, label_starts, label_bytes) -> "GBWT":
        """Node labels for an index built from parts (the Graph half of a GBZ): label i = bytes[starts[i]:starts[i+1]]."""
        starts = _u64(label_starts)
        data = np.ascontiguousarray(np.frombuffer(bytes(label_bytes), dtype=np.uint8)) if not isinstance(label_bytes, np.ndarray) \
            else np.ascontiguousarray(label_bytes, dtype=np.uint8)
        if len(starts) == 0 or int(starts[-1]) != data.nbytes:
            raise ValueError("label_starts must hold one entry per label plus the total length")
        self._check(_lib.gbwt_b200_index_attach_graph(self._h, len(starts) - 1, _ptr(starts), _ptr(data)))
        return self

    def serialize(self, gbz: bool = False) -> bytes:
        """GBWT::serialize (src/gbwt.rs:388-400) / GBZ::serialize (src/gbz.rs:662-671): the index as a Simple-SDS image,
        with the tags, DA samples, metadata and (gbz=True) the Graph it was loaded with."""
        image, n = C.c_void_p(), C.c_size_t(0)
        fn = _lib.gbwt_b200_index_serialize_gbz if gbz else _lib.gbwt_b200_index_serialize
        self._check(fn(self._h, C.byref(image), C.byref(n)))
        try:
            return bytes((C.c_uint8 * n.value).from_address(image.value)) if n.value else b""
        finally:
            _lib.gbwt_b200_free(image)

    def export_ipc(self) -> bytes:
        """Describes this index for the other processes of the node (gbwt_b200_index_export_ipc): they get their own copy on
        their own GPU with GBWT.import_ipc, copied device to device. Keep this index alive until they are done."""
        blob, n = C.c_void_p(), C.c_size_t(0)
        self._check(_lib.gbwt_b200_index_export_ipc(self._h, C.byref(blob), C.byref(n)))
        try:
            return bytes((C.c_uint8 * n.value).from_address(blob.value))
        finally:
            _lib.gbwt_b200_free(blob)

    @classmethod
    def import_ipc(cls, blob: bytes, device: int = 0) -> "GBWT":
        buf = np.frombuffer(blob, dtype=np.uint8)
        h = C.c_void_p()
        cls._check(_lib.gbwt_b200_index_import_ipc(_ptr(buf), len(buf), device, C.byref(h)))
        return cls(h.value)

    def save(self, path, gbz: bool = False) -> None:
        fn = _lib.gbwt_b200_index_save_gbz_file if gbz else _lib.gbwt_b200_index_save_file
        self._check(fn(self._h, os.fsencode(path)))

    def close(self):
        if getattr(self, "_h", None):
            _lib.gbwt_b200_index_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- statistics (src/gbwt.rs:105-175) --
    def len(self) -> int: return _lib.gbwt_b200_len(self._h)
    def is_empty(self) -> bool: return self.len() == 0
    def sequences(self) -> int: return _lib.gbwt_b200_sequences(self._h)
    def alphabet_size(self) -> int: return _lib.gbwt_b200_alphabet_size(self._h)
    def alphabet_offset(self) -> int: return _lib.gbwt_b200_alphabet_offset(self._h)
    def effective_size(self) -> int: return _lib.gbwt_b200_effective_size(self._h)
    def first_node(self) -> int: return _lib.gbwt_b200_first_node(self._h)
    def node_to_record(self, node_id: int) -> int: return node_id - self.alphabet_offset()
    def record_to_node(self, record_id: int) -> int: return record_id + self.alphabet_offset()
    def has_node(self, node_id: int) -> bool: return bool(_lib.gbwt_b200_has_node(self._h, node_id))
    def is_bidirectional(self) -> bool: return bool(_lib.gbwt_b200_is_bidirectional(self._h))
    def device(self) -> int: return _lib.gbwt_b200_device(self._h)

    def device_bytes(self) -> dict:
        b = np.zeros(10, dtype=np.uint64)
        total = _lib.gbwt_b200_device_bytes(self._h, _ptr(b))
        keys = ["descriptors", "bodies", "edges", "endmarker", "records_empty", "records_single", "records_dense",
                "records_run8", "records_run32", "records_run64"]
        out = {k: int(v) for k, v in zip(keys, b)}
        out["skips"] = int(_lib.gbwt_b200_skip_bytes(self._h))
        out["records_run_checkpointed"] = int(_lib.gbwt_b200_run_checkpoint_records(self._h))
        out["records_dense4"] = int(_lib.gbwt_b200_dense4_records(self._h))
        out["labels"] = int(_lib.gbwt_b200_graph_bytes(self._h))
        out["total"] = int(total)
        return out

    # -- unidirectional search (src/gbwt.rs:269-304) --
    def find(self, node):
        if _is_scalar(node):
            return _state_obj(self.find(np.array([node], dtype=np.uint64))[0])
        nodes = _u64(node)
        out = np.zeros(len(nodes), STATE_DTYPE)
        self._check(_lib.gbwt_b200_find(self._h, _ptr(nodes), len(nodes), _ptr(out)))
        return out

    def extend(self, state, node):
        if isinstance(state, SearchState):
            st = np.array([_state_rec(state)], dtype=STATE_DTYPE)
            return _state_obj(self.extend(st, np.array([node], dtype=np.uint64))[0])
        states = np.ascontiguousarray(state, dtype=STATE_DTYPE)
        nodes = _u64(node)
        out = np.zeros(len(nodes), STATE_DTYPE)
        self._check(_lib.gbwt_b200_extend(self._h, _ptr(states), _ptr(nodes), len(nodes), _ptr(out)))
        return out

    def find_extend(self, patterns) -> np.ndarray:
        """find(p[0]) then extend over p[1:], for an (n, k) array of patterns (src/bin/benchmark.rs:161-167)."""
        patterns = _u64(patterns)
        if patterns.ndim == 1:
            patterns = patterns.reshape(1, -1)
        n, k = patterns.shape
        out = np.zeros(n, STATE_DTYPE)
        self._check(_lib.gbwt_b200_find_extend(self._h, _ptr(patterns), n, k, _ptr(out)))
        return out

    def find_extend_u32(self, patterns) -> np.ndarray:
        """find_extend for patterns held as 32-bit node identifiers (same results, half the bytes over PCIe)."""
        patterns = np.ascontiguousarray(patterns, dtype=np.uint32)
        if patterns.ndim == 1:
            patterns = patterns.reshape(1, -1)
        n, k = patterns.shape
        out = np.zeros(n, STATE_DTYPE)
        self._check(_lib.gbwt_b200_find_extend_u32(self._h, _ptr(patterns), n, k, _ptr(out)))
        return out

    def find_extend_ragged(self, nodes, offsets) -> np.ndarray:
        nodes, offsets = _u64(nodes), _u64(offsets)
        n = len(offsets) - 1
        out = np.zeros(n, STATE_DTYPE)
        self._check(_lib.gbwt_b200_find_extend_ragged(self._h, _ptr(nodes), _ptr(offsets), n, _ptr(out)))
        return out

    # -- bidirectional search (src/gbwt.rs:311-384) --
    def bd_find(self, node):
        if _is_scalar(node):
            return _bd_obj(self.bd_find(np.array([node], dtype=np.uint64))[0])
        nodes = _u64(node)
        out = np.zeros(len(nodes), BDSTATE_DTYPE)
        self._check(_lib.gbwt_b200_bd_find(self._h, _ptr(nodes), len(nodes), _ptr(out)))
        return out

    def _bd_extend(self, fn, state, node):
        if isinstance(state, BidirectionalState):
            st = np.array([(_state_rec(state.forward), _state_rec(state.reverse))], dtype=BDSTATE_DTYPE)
            return _bd_obj(self._bd_extend(fn, st, np.array([node], dtype=np.uint64))[0])
        states = np.ascontiguousarray(state, dtype=BDSTATE_DTYPE)
        nodes = _u64(node)
        out = np.zeros(len(nodes), BDSTATE_DTYPE)
        self._check(fn(self._h, _ptr(states), _ptr(nodes), len(nodes), _ptr(out)))
        return out

    def extend_forward(self, state, node):
        return self._bd_extend(_lib.gbwt_b200_extend_forward, state, node)

    def extend_backward(self, state, node):
        return self._bd_extend(_lib.gbwt_b200_extend_backward, state, node)

    def bd_search(self, nodes, offsets, first, start, end) -> np.ndarray:
        """Fused bd_find + extend_forward* + extend_backward* (the driver of src/gbwt/tests.rs:352-361)."""
        nodes, offsets, first, start, end = map(_u64, (nodes, offsets, first, start, end))
        n = len(first)
        out = np.zeros(n, BDSTATE_DTYPE)
        self._check(_lib.gbwt_b200_bd_search(self._h, _ptr(nodes), _ptr(offsets), _ptr(first), _ptr(start), _ptr(end), n, _ptr(out)))
        return out

    def follow(self, states, backward: bool = False):
        """All non-empty single-node extensions of each state (GBZ::follow_forward / follow_backward,
        src/gbz.rs:519-544): returns (offsets, extensions, counts), counts[i] = 2^64-1 where the reference is None."""
        states = np.ascontiguousarray(states, dtype=BDSTATE_DTYPE)
        n = len(states)
        counts = np.zeros(n, np.uint64)
        self._check(_lib.gbwt_b200_follow(self._h, _ptr(states), n, int(backward), None, None, _ptr(counts)))
        sizes = np.where(counts == _U64MAX, np.uint64(0), counts)
        offsets = np.zeros(n + 1, np.uint64)
        np.cumsum(sizes, out=offsets[1:])
        out = np.zeros(int(offsets[-1]), BDSTATE_DTYPE)
        self._check(_lib.gbwt_b200_follow(self._h, _ptr(states), n, int(backward), _ptr(offsets), _ptr(out), _ptr(counts)))
        return offsets, out, counts

    def follow_forward(self, state):
        """GBZ::follow_forward for one state: list of BidirectionalState, or None."""
        return self._follow_one(state, False)

    def follow_backward(self, state):
        return self._follow_one(state, True)

    def _follow_one(self, state: "BidirectionalState", backward: bool):
        st = np.array([(_state_rec(state.forward), _state_rec(state.reverse))], dtype=BDSTATE_DTYPE)
        _, out, counts = self.follow(st, backward)
        if counts[0] == _U64MAX:
            return None
        return [_bd_obj(o) for o in out]

    # -- sequence navigation (src/gbwt.rs:213-261) --
    def start(self, seq_id):
        if _is_scalar(seq_id):
            r = self.start(np.array([seq_id], dtype=np.uint64))[0]
            return Pos(int(r["node"]), int(r["offset"])) if r["node"] != ENDMARKER else None
        ids = _u64(seq_id)
        out = np.zeros(len(ids), POS_DTYPE)
        self._check(_lib.gbwt_b200_start(self._h, _ptr(ids), len(ids), _ptr(out)))
        return out

    def _step(self, fn, pos):
        if isinstance(pos, Pos):
            r = self._step(fn, np.array([(pos.node, pos.offset)], dtype=POS_DTYPE))[0]
            return Pos(int(r["node"]), int(r["offset"])) if r["node"] != ENDMARKER else None
        positions = np.ascontiguousarray(pos, dtype=POS_DTYPE)
        out = np.zeros(len(positions), POS_DTYPE)
        self._check(fn(self._h, _ptr(positions), len(positions), _ptr(out)))
        return out

    def forward(self, pos):
        return self._step(_lib.gbwt_b200_forward, pos)

    def backward(self, pos):
        return self._step(_lib.gbwt_b200_backward, pos)

    def sequence_lengths(self, seq_ids) -> np.ndarray:
        ids = _u64(seq_ids)
        out = np.zeros(len(ids), np.uint64)
        self._check(_lib.gbwt_b200_sequence_lengths(self._h, _ptr(ids), len(ids), _ptr(out)))
        return out

    def extract(self, seq_ids, lengths=None):
        """GBWT::sequence(id).collect() for many ids: returns (offsets, nodes, lengths)."""
        ids = _u64(seq_ids)
        if lengths is None:
            lengths = self.sequence_lengths(ids)
        sizes = np.where(lengths == _U64MAX, np.uint64(0), lengths)
        offsets = np.zeros(len(ids) + 1, np.uint64)
        np.cumsum(sizes, out=offsets[1:])
        nodes = np.zeros(int(offsets[-1]), np.uint64)
        got = np.zeros(len(ids), np.uint64)
        self._check(_lib.gbwt_b200_extract(self._h, _ptr(ids), len(ids), _ptr(offsets), _ptr(nodes), _ptr(got)))
        return offsets, nodes, got

    def sequence(self, seq_id: int) -> Optional[Iterator[int]]:
        """GBWT::sequence (src/gbwt.rs:253-261): an iterator over the node ids, or None if id >= sequences()."""
        if seq_id >= self.sequences():
            return None
        _, nodes, _ = self.extract(np.array([seq_id], dtype=np.uint64))
        return iter(int(x) for x in nodes)

    # -- locate: which sequences, and where (beyond the crate; the C++ GBWT's locate is the model, gbwt_b200.h) --
    def locate(self, what):
        """A Pos: (sequence, index) of the position -- node number `index` of GBWT::sequence(sequence) -- or None where there
        is no such position. A SearchState: the list of (sequence, index) of its positions in offset order (empty for None).
        The C++ GBWT's locate(state) is sorted(set(s for s, _ in ...)). Needs an index created with locate=True."""
        if isinstance(what, Pos):
            r = self.locate_positions(np.array([(what.node, what.offset)], dtype=POS_DTYPE))[0]
            return None if r["sequence"] == _U64MAX else (int(r["sequence"]), int(r["index"]))
        if isinstance(what, SearchState):
            _, occ = self.locate_states(np.array([_state_rec(what)], dtype=STATE_DTYPE))
            return [(int(o["sequence"]), int(o["index"])) for o in occ]
        if what is None:
            return []
        raise TypeError("locate takes a Pos or a SearchState")

    def locate_positions(self, positions) -> np.ndarray:
        """locate for many positions: a structured array of (sequence, index), UINT64_MAX in both where there is none."""
        positions = np.ascontiguousarray(positions, dtype=POS_DTYPE)
        out = np.zeros(len(positions), OCCURRENCE_DTYPE)
        self._check(_lib.gbwt_b200_locate(self._h, _ptr(positions), len(positions), _ptr(out)))
        return out

    def locate_states(self, states):
        """The occurrences of many search states: (offsets, occurrences), those of state i at occurrences[offsets[i]:offsets[i+1]],
        in offset order (shaped like extract)."""
        states = np.ascontiguousarray(states, dtype=STATE_DTYPE)
        n = len(states)
        sizes = np.where(states["end"] > states["start"], states["end"] - states["start"], np.uint64(0)).astype(np.uint64)
        offsets = np.zeros(n + 1, np.uint64)
        np.cumsum(sizes, out=offsets[1:])
        out = np.zeros(int(offsets[-1]), OCCURRENCE_DTYPE)
        counts = np.zeros(n, np.uint64)
        self._check(_lib.gbwt_b200_locate_states(self._h, _ptr(states), n, _ptr(offsets), _ptr(out), _ptr(counts)))
        assert np.array_equal(counts, sizes)
        return offsets, out

    def locate_device(self, d_positions: int, n: int, d_out: int, stream: int = 0):
        self._check(_lib.gbwt_b200_locate_device(self._h, d_positions, n, d_out, stream))

    def locate_states_device(self, d_states: int, n: int, d_out_offsets: int, d_out: int, d_counts: int = 0, stream: int = 0):
        self._check(_lib.gbwt_b200_locate_states_device(self._h, d_states, n, d_out_offsets or None, d_out or None, d_counts or None, stream))

    def locate_info(self) -> dict:
        """Locate samples (gbwt_b200_locate_info); lf_steps is only counted with GBWT_B200_LOCATE_STATS=1."""
        raw = np.zeros(6, dtype=np.uint64)
        _lib.gbwt_b200_locate_info(self._h, _ptr(raw))
        keys = ("present", "interval", "samples", "bytes", "build_us", "lf_steps")
        return {k: int(v) for k, v in zip(keys, raw)}

    # -- ranges of sequences (beyond the crate; include/gbwt_b200_ranges.h) --
    def seek(self, seq_ids, indexes=None):
        """Position of node number j of GBWT::sequence(s) (start(s) and j forward steps). seek(s, j) returns a Pos or None;
        with arrays, a POS_DTYPE array ({0, 0} where s >= sequences() or j >= the length of s)."""
        if _is_scalar(seq_ids):
            r = self.seek(np.array([seq_ids], dtype=np.uint64), np.array([indexes], dtype=np.uint64))[0]
            return Pos(int(r["node"]), int(r["offset"])) if r["node"] != ENDMARKER else None
        ids, idx = _u64(seq_ids), _u64(indexes)
        if len(ids) != len(idx):
            raise ValueError("seq_ids and indexes must have the same length")
        out = np.zeros(len(ids), POS_DTYPE)
        self._check(_lib.gbwt_b200_seek(self._h, _ptr(ids), _ptr(idx), len(ids), _ptr(out)))
        return out

    def _ranges(self, fn, full, seq_ids, starts, ends, dtype):
        ids, starts, ends = _u64(seq_ids), _u64(starts), _u64(ends)
        if not len(ids) == len(starts) == len(ends):
            raise ValueError("seq_ids, starts and ends must have the same length")
        full = np.where(full == _U64MAX, np.uint64(0), full)
        stop = np.minimum(ends, full)
        sizes = np.where(stop > starts, stop - starts, np.uint64(0)).astype(np.uint64)
        offsets = np.zeros(len(ids) + 1, np.uint64)
        np.cumsum(sizes, out=offsets[1:])
        data = np.zeros(int(offsets[-1]), dtype)
        got = np.zeros(len(ids), np.uint64)
        self._check(fn(self._h, _ptr(ids), _ptr(starts), _ptr(ends), len(ids), _ptr(offsets), _ptr(data), _ptr(got)))
        return offsets, data, got

    def extract_ranges(self, seq_ids, starts, ends):
        """extract(s)[start:min(end, len)] for many (s, start, end): (offsets, nodes, lengths) shaped like extract; lengths[i] =
        max(0, min(end, len) - start), UINT64_MAX where the sequence is None."""
        return self._ranges(_lib.gbwt_b200_extract_ranges, self.sequence_lengths(seq_ids), seq_ids, starts, ends, np.uint64)

    def extract_dna_ranges(self, seq_ids, starts, ends):
        """Bytes [start, min(end, L)) of extract_dna(s) without its endmarker (L = dna_lengths(s) - 1), for many (s, start, end):
        (offsets, bytes, lengths) shaped like extract_dna."""
        full = self.dna_lengths(seq_ids)
        full = np.where(full == _U64MAX, full, full - np.uint64(1))
        return self._ranges(_lib.gbwt_b200_extract_dna_ranges, full, seq_ids, starts, ends, np.uint8)

    def seek_device(self, d_ids: int, d_indexes: int, n: int, d_out: int, stream: int = 0):
        self._check(_lib.gbwt_b200_seek_device(self._h, d_ids, d_indexes, n, d_out, stream))

    def extract_ranges_device(self, d_ids: int, d_starts: int, d_ends: int, m: int, d_out_offsets: int, d_nodes: int, d_lengths: int,
                              stream: int = 0):
        self._check(_lib.gbwt_b200_extract_ranges_device(self._h, d_ids, d_starts, d_ends, m, d_out_offsets, d_nodes, d_lengths, stream))

    def extract_dna_ranges_device(self, d_ids: int, d_starts: int, d_ends: int, m: int, d_out_offsets: int, d_bytes: int, d_lengths: int,
                                  stream: int = 0):
        self._check(_lib.gbwt_b200_extract_dna_ranges_device(self._h, d_ids, d_starts, d_ends, m, d_out_offsets, d_bytes, d_lengths, stream))

    # -- node sequences and DNA-level extraction (GBZ files; src/gbz.rs:286-306, src/bin/gbz-extract.rs:173-189) --
    def has_graph(self) -> bool: return bool(_lib.gbwt_b200_has_graph(self._h))
    def graph_sequences(self) -> int: return _lib.gbwt_b200_graph_sequences(self._h)

    def node_sequence_lengths(self, node_ids) -> np.ndarray:
        ids = _u64(node_ids)
        out = np.zeros(len(ids), np.uint64)
        self._check(_lib.gbwt_b200_node_sequence_lengths(self._h, _ptr(ids), len(ids), _ptr(out)))
        return out

    def node_sequences(self, node_ids):
        """GBZ::sequence for many original-graph node ids: (offsets, bytes, lengths); UINT64_MAX length = None."""
        ids = _u64(node_ids)
        lengths = self.node_sequence_lengths(ids)
        offsets = np.zeros(len(ids) + 1, np.uint64)
        np.cumsum(np.where(lengths == _U64MAX, np.uint64(0), lengths), out=offsets[1:])
        data = np.zeros(int(offsets[-1]), np.uint8)
        got = np.zeros(len(ids), np.uint64)
        self._check(_lib.gbwt_b200_node_sequences(self._h, _ptr(ids), len(ids), _ptr(offsets), _ptr(data), _ptr(got)))
        return offsets, data, got

    def sequence_len(self, node_id: int) -> Optional[int]:
        """GBZ::sequence_len (src/gbz.rs:301-306)."""
        n = int(self.node_sequence_lengths([node_id])[0])
        return None if n == int(_U64MAX) else n

    def node_sequence(self, node_id: int) -> Optional[bytes]:
        """GBZ::sequence (src/gbz.rs:292-298)."""
        _, data, got = self.node_sequences([node_id])
        return None if got[0] == _U64MAX else data.tobytes()

    def dna_lengths(self, seq_ids) -> np.ndarray:
        ids = _u64(seq_ids)
        out = np.zeros(len(ids), np.uint64)
        self._check(_lib.gbwt_b200_dna_lengths(self._h, _ptr(ids), len(ids), _ptr(out)))
        return out

    def extract_dna(self, seq_ids, endmarker: int = 0, lengths=None):
        """extract_sequence of gbz-extract for many GBWT sequence ids: (offsets, bytes, lengths)."""
        ids = _u64(seq_ids)
        if lengths is None:
            lengths = self.dna_lengths(ids)
        offsets = np.zeros(len(ids) + 1, np.uint64)
        np.cumsum(np.where(lengths == _U64MAX, np.uint64(0), lengths), out=offsets[1:])
        data = np.zeros(int(offsets[-1]), np.uint8)
        got = np.zeros(len(ids), np.uint64)
        self._check(_lib.gbwt_b200_extract_dna(self._h, _ptr(ids), len(ids), endmarker, _ptr(offsets), _ptr(data), _ptr(got)))
        return offsets, data, got

    def path_dna(self, seq_id: int, endmarker: int = 0) -> Optional[bytes]:
        """extract_sequence(gbz, path_id, orientation) with seq_id = encode_path(path_id, orientation); None if no such path."""
        if seq_id >= self.sequences():
            return None
        _, data, _ = self.extract_dna([seq_id], endmarker)
        return data.tobytes()

    def dna_lengths_device(self, d_ids: int, m: int, d_lengths: int, stream: int = 0):
        self._check(_lib.gbwt_b200_dna_lengths_device(self._h, d_ids, m, d_lengths, stream))

    def extract_dna_device(self, d_ids: int, m: int, endmarker: int, d_out_offsets: int, d_bytes: int, d_lengths: int, stream: int = 0):
        self._check(_lib.gbwt_b200_extract_dna_device(self._h, d_ids, m, endmarker, d_out_offsets, d_bytes, d_lengths, stream))

    def checkpoint_info(self) -> dict:
        raw = np.zeros(6, dtype=np.uint64)
        _lib.gbwt_b200_checkpoint_info(self._h, _ptr(raw))
        keys = ("present", "interval", "entries", "bytes", "build_us", "max_segments")
        return {k: int(v) for k, v in zip(keys, raw)}

    def window_info(self) -> dict:
        """Plan and counters of the record-window search kernel (gbwt_b200_window_info)."""
        raw = np.zeros(14, dtype=np.uint64)
        _lib.gbwt_b200_window_info(self._h, _ptr(raw))
        keys = ("can_run", "default", "window_records", "margin", "body_units", "threads", "smem_bytes", "windows",
                "edges", "edges_local", "queries", "deferred", "kernel_ns", "launches")
        return {k: int(v) for k, v in zip(keys, raw)}

    # -- device-pointer entry points (raw addresses, e.g. torch.Tensor.data_ptr(); stream = cudaStream_t) --
    def find_extend_device(self, d_patterns: int, n: int, k: int, d_out: int, stream: int = 0):
        self._check(_lib.gbwt_b200_find_extend_device(self._h, d_patterns, n, k, d_out, stream))

    def find_extend_u32_device(self, d_patterns: int, n: int, k: int, d_out: int, stream: int = 0):
        self._check(_lib.gbwt_b200_find_extend_u32_device(self._h, d_patterns, n, k, d_out, stream))

    def bd_search_device(self, d_nodes, d_offsets, d_first, d_start, d_end, n, d_out, stream: int = 0):
        self._check(_lib.gbwt_b200_bd_search_device(self._h, d_nodes, d_offsets, d_first, d_start, d_end, n, d_out, stream))

    def sequence_lengths_device(self, d_ids: int, m: int, d_lengths: int, stream: int = 0):
        self._check(_lib.gbwt_b200_sequence_lengths_device(self._h, d_ids, m, d_lengths, stream))

    def extract_device(self, d_ids: int, m: int, d_out_offsets: int, d_nodes: int, d_lengths: int, stream: int = 0):
        self._check(_lib.gbwt_b200_extract_device(self._h, d_ids, m, d_out_offsets, d_nodes, d_lengths, stream))


# ---- building a GBWT from paths (beyond the crate; include/gbwt_b200_build.h) --

def _paths_arrays(paths):
    """(nodes, offsets) as uint64 arrays from a list of paths or from a (nodes, offsets) pair."""
    if isinstance(paths, tuple) and len(paths) == 2 and isinstance(paths[1], np.ndarray):
        return _u64(paths[0]), _u64(paths[1])
    lengths = [len(p) for p in paths]
    offsets = np.zeros(len(lengths) + 1, np.uint64)
    np.cumsum(np.array(lengths, dtype=np.uint64), out=offsets[1:])
    nodes = np.concatenate([_u64(p) for p in paths]) if offsets[-1] else np.zeros(0, np.uint64)
    return nodes, offsets


def _take_image(call, info):
    image, n = C.c_void_p(), C.c_size_t(0)
    stats = np.zeros(4, np.uint64)
    GBWT._check(call(C.byref(image), C.byref(n), _ptr(stats)))
    try:
        out = bytes((C.c_uint8 * n.value).from_address(image.value))
    finally:
        _lib.gbwt_b200_free(image)
    if info is not None:
        info.update(positions=int(stats[0]), rounds=int(stats[1]), device_us=int(stats[2]), peak_device_bytes=int(stats[3]))
    return out


def build_image(paths, bidirectional: bool = True, device: int = 0, info: Optional[dict] = None) -> bytes:
    """The Simple-SDS GBWT file of the paths, built on the device: a list of paths (sequences of GBWT node ids) or a
    (nodes, offsets) pair with path q = nodes[offsets[q]:offsets[q+1]]. bidirectional: sequences 2q = path q and 2q+1 = its
    reverse with every node flipped. `info`, a dict, receives positions, rounds, device_us and peak_device_bytes."""
    nodes, offsets = _paths_arrays(paths)
    n = max(len(offsets) - 1, 0)
    return _take_image(lambda img, ln, st: _lib.gbwt_b200_build_image(
        _ptr(nodes) if len(nodes) else None, _ptr(offsets) if len(offsets) else None, n, int(bidirectional), device, img, ln, st), info)


def build_image_device(nodes, offsets, n: Optional[int] = None, bidirectional: bool = True, device: int = 0, stream=0,
                       info: Optional[dict] = None) -> bytes:
    """build_image from device arrays: torch tensors (int64 / uint64 on the device) or raw addresses, read on `stream`
    (a torch.cuda.Stream or a cudaStream_t address). Offsets are absolute; n = the number of paths (len(offsets) - 1 for a
    tensor)."""
    def addr(x):
        if hasattr(x, "data_ptr"):
            if x.element_size() != 8 or not x.is_contiguous():
                raise ValueError("nodes and offsets must be contiguous 64-bit tensors")
            return x.data_ptr()
        return x or None
    if n is None:
        n = len(offsets) - 1
    s = getattr(stream, "cuda_stream", stream) or None
    return _take_image(lambda img, ln, st: _lib.gbwt_b200_build_image_device(
        addr(nodes), addr(offsets), n, int(bidirectional), device, s, img, ln, st), info)


from .distributed import gather_states, shard_range  # noqa: E402,F401
