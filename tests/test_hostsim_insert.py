"""The insertion walk of gbwt-rs_b200/csrc/insert_step.h run on the CPU over the product's device layout of an index A, and
the record merge of insert.cu restated in Python. CPU only; tests/hostsim is test infrastructure, not a fallback.

- alpha(e), the A entries of e's record that sort before a new entry e, from the shared step function, must equal a
  brute-force count over the sort keys of tests/gbwt_builder.py (reversed prefix, then the sequence id).
- Step 3 of the insertion (alpha and beta -> records with merged edges and maximal runs), fed from the builder and the walk,
  must give the records of build_bwt(seqs(A) + S)."""
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
LAYOUT_AUTO, LAYOUT_RUNS = 0, 1
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        tmp = tempfile.mkdtemp(prefix="gbwt_hostsim_insert_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libhostsim_insert.so")
        csrc = os.path.join(ROOT, "gbwt-rs_b200", "csrc")
        subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-fopenmp", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", out,
                        os.path.join(HERE, "hostsim", "hostsim_insert.cpp"), os.path.join(csrc, "layout_builder.cpp"),
                        os.path.join(csrc, "sds_loader.cpp"), "-ldl"], check=True, capture_output=True)
        L = C.CDLL(out)
        p = C.c_void_p
        L.hi_load.restype, L.hi_load.argtypes = p, [p, C.c_size_t, C.c_int, C.c_char_p, C.c_size_t]
        L.hi_free.argtypes = [p]
        L.hi_alpha.argtypes = [p, p, p, C.c_size_t, p]
        L.hi_before.argtypes = [p, p, p, C.c_size_t, p]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Sim:
    def __init__(self, image, policy):
        arr = np.frombuffer(bytes(image), dtype=np.uint8)
        err = C.create_string_buffer(256)
        self.h = lib().hi_load(_p(arr), arr.nbytes, policy, err, 256)
        assert self.h, err.value.decode()

    def __del__(self):
        if getattr(self, "h", None):
            lib().hi_free(self.h)

    def alpha(self, seqs):
        """alpha of every node of every new sequence, per sequence."""
        lengths = [len(s) for s in seqs]
        offsets = np.zeros(len(seqs) + 1, np.uint64)
        np.cumsum(np.array(lengths, dtype=np.uint64), out=offsets[1:])
        nodes = np.array([x for s in seqs for x in s] or [0], dtype=np.uint64)
        out = np.zeros(max(int(offsets[-1]), 1), np.uint64)
        lib().hi_alpha(self.h, _p(nodes), _p(offsets), len(seqs), _p(out))
        return [[int(x) for x in out[offsets[q]:offsets[q + 1]]] for q in range(len(seqs))]


def visits(seqs, first_id=0):
    """record node -> [(key, successor, (sequence, index))] sorted by key; index -1 is the entry in record 0."""
    out = {}
    for j, s in enumerate(seqs):
        sid = first_id + j
        out.setdefault(0, []).append(((sid,), s[0] if s else 0, (j, -1)))
        for k, v in enumerate(s):
            out.setdefault(v, []).append((tuple(reversed(s[:k])) + (0, sid), s[k + 1] if k + 1 < len(s) else 0, (j, k)))
    for lst in out.values():
        lst.sort(key=lambda t: t[0])
    return out


def brute_alpha(a_seqs, new_seqs):
    a_vis = visits(a_seqs)
    new_vis = visits(new_seqs, len(a_seqs))
    alpha = [[None] * len(s) for s in new_seqs]
    for v, lst in new_vis.items():
        keys = [t[0] for t in a_vis.get(v, [])]
        for key, _, (j, k) in lst:
            if k >= 0:
                alpha[j][k] = sum(1 for x in keys if x < key)
    return alpha


def before(vis, v, w):
    """Entries of record v whose predecessor is below w (the predecessor is the key's first element; 0 = the endmarker)."""
    return sum(1 for key, _, _ in vis.get(v, []) if (key[0] if len(key) > 2 else 0) < w)


def merge_records(a_seqs, new_seqs, alpha):
    """Step 3 of the insertion: A's records and the new entries in beta order (from the builder), alpha from the walk ->
    (offset, alphabet_size, records) in the form of gbwt_builder.build_records."""
    a_vis, s_vis = visits(a_seqs), visits(new_seqs, len(a_seqs))
    nodes = [v for v in list(a_vis) + list(s_vis) if v != 0]
    if not nodes:
        return None
    offset, alphabet_size = min(nodes) - 1, max(nodes) + 1
    records = []
    for r in range(alphabet_size - offset):
        w = 0 if r == 0 else r + offset
        a_succ = [succ for _, succ, _ in a_vis.get(w, [])]
        s_entries = [(len(a_seqs) if k < 0 else alpha[j][k], succ) for _, succ, (j, k) in s_vis.get(w, [])]
        merged, i = [], 0
        for al, succ in s_entries:  # beta order; alpha is non-decreasing along it
            merged += a_succ[i:al]
            i = max(i, al)
            merged.append(succ)
        merged += a_succ[i:]
        if not merged:
            records.append(([], []))
            continue
        succs = sorted(set(merged))
        edges = [(v, 0 if v == 0 else before(a_vis, v, w) + before(s_vis, v, w)) for v in succs]
        rank = {v: x for x, v in enumerate(succs)}
        runs = []
        for v in merged:
            if runs and runs[-1][0] == rank[v]:
                runs[-1][1] += 1
            else:
                runs.append([rank[v], 1])
        records.append((edges, [tuple(x) for x in runs]))
    return offset, alphabet_size, records


def new_paths(rng, a_paths, lo, hi):
    """Paths for S: copies, prefixes and extensions of A's paths, empty and single-node paths, nodes A lacks below and above
    its range, and new edges between A's nodes."""
    walk = lambda n: [2 * rng.randint(lo, hi) + (1 if rng.random() < 0.3 else 0) for _ in range(n)]
    out = [walk(rng.randint(1, 8)) for _ in range(rng.randint(1, 6))]
    if a_paths:
        p = list(rng.choice(a_paths))
        out += [p, p[:rng.randint(0, len(p))], p + walk(3), walk(2) + p]
    out += [[], [2 * hi + 2], [max(2, 2 * lo - 2)], [2 * hi + 6, 2 * lo, 2 * hi + 6]]
    rng.shuffle(out)
    return out


def sequences_of(g):
    return [[int(x) for x in g.sequence(i)] for i in range(g.sequences())]


def cases():
    for name in FIXTURES:
        yield name, (lambda name=name: (open(os.path.join(GOLDEN, name), "rb").read(), None))
    for seed in range(6):
        for bidirectional in (True, False):
            yield f"random-{seed}-{bidirectional}", (lambda seed=seed, b=bidirectional: random_graph(seed, b))


CASES = list(cases())


@pytest.mark.parametrize("policy", [LAYOUT_AUTO, LAYOUT_RUNS])
@pytest.mark.parametrize("case", [c[0] for c in CASES])
def test_alpha_against_brute_force_keys(case, policy):
    image, _ = dict(CASES)[case]()
    g = orc.GBWT.load(image)
    a_seqs = sequences_of(g)
    bidirectional = g.is_bidirectional()
    a_paths = a_seqs[0::2] if bidirectional else a_seqs
    nodes = [x // 2 for s in a_seqs for x in s] or [1]
    rng = random.Random(case + str(policy))
    sim = Sim(image, policy)
    for _ in range(4):
        paths = [p for p in new_paths(rng, a_paths, max(1, min(nodes) - 2), max(nodes) + 2) if len(p) < 40]
        s = gb.bidirectional_sequences(paths) if bidirectional else paths
        got = sim.alpha(s)
        assert got == brute_alpha(a_seqs, s)
        want = gb.build_records(a_seqs + s)
        assert merge_records(a_seqs, s, got) == want


def test_before_counts_entries_with_a_smaller_predecessor():
    image, paths = random_graph(3, True)
    g = orc.GBWT.load(image)
    a_seqs = sequences_of(g)
    vis = visits(a_seqs)
    nodes = sorted(v for v in vis if v != 0)
    vs = np.array([v for v in nodes for _ in range(len(nodes) + 3)], dtype=np.uint64)
    ws = np.array([w for _ in nodes for w in [0] + nodes + [nodes[-1] + 1, nodes[-1] + 7]], dtype=np.uint64)
    out = np.zeros(len(vs), np.uint64)
    sim = Sim(image, LAYOUT_AUTO)
    lib().hi_before(sim.h, _p(vs), _p(ws), len(vs), _p(out))
    for v, w, x in zip(vs, ws, out):
        assert int(x) == before(vis, int(v), int(w)), (v, w)
