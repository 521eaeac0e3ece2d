"""Ranges of sequences (include/gbwt_b200_ranges.h) against slices of the oracle: seek(s, j) is start(s) and j forward steps,
a node range is a slice of GBWT::sequence(s), a DNA range a slice of extract_dna(s) without its endmarker."""
import os
import random
import re

import numpy as np
import pytest

import gbwt_builder as gb
from locate_oracle import pattern_origins
from oracle import oracle as orc
from synth import synth
from test_gpu_dna import image_args, random_labels
from test_hostsim_ranges import paths_of
from test_oracle_locate import FIXTURES, GOLDEN, random_graph

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U64MAX = 2**64 - 1
SENTINEL = 0xAB


@pytest.fixture(scope="module")
def b200():
    import gbwt_rs_b200
    return gbwt_rs_b200


def index(b200, image, monkeypatch, shift=None, checkpoints=True, **kw):
    """An index with path checkpoints every 2^shift nodes (None: the default interval), or without any."""
    monkeypatch.setenv("GBWT_B200_CHECKPOINTS", "1" if checkpoints else "0")
    if shift is None:
        monkeypatch.delenv("GBWT_B200_CHECKPOINT_SHIFT", raising=False)
    else:
        monkeypatch.setenv("GBWT_B200_CHECKPOINT_SHIFT", str(shift))
    e = b200.GBWT.from_bytes(image, **kw)
    assert bool(e.checkpoint_info()["present"]) == checkpoints
    return e


# ---- truth -------------------------------------------------------------------------------------------------------------

def sequences_of(g):
    return [np.asarray(g.sequence(s), np.uint64) for s in range(g.sequences())]


def edge_ranges(lengths, interval, rng, n_random=200):
    """(ids, starts, ends): whole sequences, empty, single-node and reversed ranges, ranges past the end, starts and ends on and
    around every multiple of the interval and the 31 nodes after it (where the checkpoints lie), long random ranges, None ids."""
    rows = []
    n = len(lengths)
    for s, L in enumerate(lengths):
        rows += [(s, 0, L), (s, 0, L + 5), (s, L, L), (s, L, L + 3), (s, L + 3, L + 9), (s, 5, 3), (s, 0, 0), (s, 0, 1), (s, 0, U64MAX)]
        if L:
            rows += [(s, L - 1, L), (s, L - 1, L + 1), (s, L // 2, L // 2 + 1), (s, L // 3, L // 3)]
        for k in range(0, L // interval + 1):
            for d in (-1, 0, 1, 31, 32, 33):
                x = k * interval + d
                if 0 <= x <= L + 1:
                    rows += [(s, x, x + 1), (s, x, min(L, x + interval + 2)), (s, max(0, x - 40), x), (s, x, L), (s, 0, x)]
    for _ in range(n_random):
        s = rng.randrange(n) if n else 0
        L = lengths[s] if n else 0
        a = rng.randint(0, L + 2)
        rows.append((s, a, a + rng.choice([0, 1, 2, 7, 64, 300, 5000, L + 10])))
    rows += [(n, 0, 5), (n + 3, 0, 0), (U64MAX, 1, 2)]
    a = np.array(rows, dtype=np.uint64)
    return a[:, 0].copy(), a[:, 1].copy(), a[:, 2].copy()


def sliced(full, ids, starts, ends, dtype):
    """What a range call returns: (offsets, data, lengths), each result sized to its clipped range."""
    parts, lengths = [], []
    for s, a, b in zip(ids.tolist(), starts.tolist(), ends.tolist()):
        if s >= len(full):
            parts.append(np.zeros(0, dtype)); lengths.append(U64MAX)
            continue
        piece = full[s][a:min(b, len(full[s]))] if a < min(b, len(full[s])) else full[s][:0]
        parts.append(np.asarray(piece, dtype)); lengths.append(len(piece))
    offsets = np.zeros(len(parts) + 1, np.uint64)
    np.cumsum([len(p) for p in parts], out=offsets[1:])
    data = np.concatenate(parts) if parts else np.zeros(0, dtype)
    return offsets, data.astype(dtype), np.array(lengths, np.uint64)


def check_node_ranges(e, seqs, ids, starts, ends):
    want = sliced(seqs, ids, starts, ends, np.uint64)
    got = e.extract_ranges(ids, starts, ends)
    for w, g_ in zip(want, got):
        assert np.array_equal(w, g_)


def dna_of(g):
    return [np.frombuffer(g.extract_dna(s)[:-1], np.uint8) for s in range(g.sequences())]


def check_dna_ranges(e, dna, ids, starts, ends):
    want = sliced(dna, ids, starts, ends, np.uint8)
    got = e.extract_dna_ranges(ids, starts, ends)
    for w, g_ in zip(want, got):
        assert np.array_equal(w, g_)


def check_seek(e, paths, extra_j=()):
    ids, idx, want = [], [], []
    for s, pos in enumerate(paths):
        for j in list(range(len(pos) + 1)) + [len(pos) + x for x in extra_j]:
            ids.append(s); idx.append(j); want.append(pos[j] if j < len(pos) else (0, 0))
    n = len(paths)
    ids += [n, n + 1, U64MAX]; idx += [0, 0, 0]; want += [(0, 0)] * 3
    got = e.seek(np.array(ids, np.uint64), np.array(idx, np.uint64))
    assert np.array_equal(got.view(np.uint64).reshape(-1, 2), np.array(want, np.uint64).reshape(-1, 2))
    if n and paths[0]:
        assert e.seek(0, 0) == e.start(0) and e.seek(0, len(paths[0])) is None


def check_all(e, g, seed, interval):
    paths = paths_of(g)
    check_seek(e, paths)
    seqs = sequences_of(g)
    check_node_ranges(e, seqs, *edge_ranges([len(x) for x in seqs], interval, random.Random(seed)))
    return paths, seqs


# ---- seek and node ranges ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("layout", ["auto", "runs"])
@pytest.mark.parametrize("name", FIXTURES)
def test_fixtures(b200, name, layout, monkeypatch):
    img = open(os.path.join(GOLDEN, name), "rb").read()
    g = orc.GBWT.load(img)
    for ckpt in (True, False):
        check_all(index(b200, img, monkeypatch, 6, ckpt, layout=layout), g, 1, 64)


@pytest.mark.parametrize("checkpoints,shift", [(True, 6), (True, 8), (False, None)])
@pytest.mark.parametrize("seed", range(4))
def test_random_graphs(b200, seed, checkpoints, shift, monkeypatch):
    img, _ = random_graph(seed, seed % 2 == 0)
    check_all(index(b200, img, monkeypatch, shift, checkpoints), orc.GBWT.load(img), seed, 1 << (shift or 6))


@pytest.mark.parametrize("checkpoints,shift", [(True, 6), (True, 8), (False, None)])
@pytest.mark.parametrize("model", [dict(), dict(alt_ppm=50_000, tri_mod=4)])
def test_bubble_chains(b200, model, checkpoints, shift, monkeypatch):
    S, H, seed = 700, 12, 5
    img = synth.bubble_chain(S, H, seed, **model)
    g = orc.GBWT.load(img.array)
    e = index(b200, img.array, monkeypatch, shift, checkpoints)
    check_all(e, g, seed, 1 << (shift or 6))
    if checkpoints:
        # ranges across many checkpoints, from everywhere
        seqs = sequences_of(g)
        rng = np.random.default_rng(seed)
        ids = rng.integers(0, len(seqs), 3000).astype(np.uint64)
        starts = rng.integers(0, 2200, 3000).astype(np.uint64)
        ends = starts + rng.integers(0, 2000, 3000).astype(np.uint64)
        check_node_ranges(e, seqs, ids, starts, ends)


def test_seek_inverts_locate(b200, monkeypatch):
    S, H, seed = 600, 10, 3
    img = synth.bubble_chain(S, H, seed)
    e = index(b200, img.array, monkeypatch, 6, locate=True)
    lengths = e.sequence_lengths(np.arange(e.sequences(), dtype=np.uint64)).astype(np.int64)
    ids = np.repeat(np.arange(len(lengths), dtype=np.uint64), lengths)
    idx = np.concatenate([np.arange(n, dtype=np.uint64) for n in lengths])
    occ = e.locate_positions(e.seek(ids, idx))
    assert np.array_equal(occ["sequence"], ids) and np.array_equal(occ["index"], idx)


# ---- DNA ranges --------------------------------------------------------------------------------------------------------

def dna_ranges(dna, rng, n=600):
    rows = []
    for s, d in enumerate(dna):
        L = len(d)
        rows += [(s, 0, L), (s, 0, L + 9), (s, L, L + 1), (s, 3, 1), (s, 0, U64MAX), (s, max(0, L - 1), L)]
    for _ in range(n):
        s = rng.randrange(len(dna))
        L = len(dna[s])
        a = rng.randint(0, L + 1)
        rows.append((s, a, a + rng.choice([0, 1, 2, 3, 17, 100, 1000, L])))
    rows += [(len(dna), 0, 4), (U64MAX, 0, 1)]
    a = np.array(rows, dtype=np.uint64)
    return a[:, 0].copy(), a[:, 1].copy(), a[:, 2].copy()


@pytest.mark.parametrize("dna_checkpoints", ["1", "0"])
@pytest.mark.parametrize("seed", range(4))
def test_dna_random_graphs(b200, seed, dna_checkpoints, monkeypatch):
    from test_hostsim_layout import random_paths
    monkeypatch.setenv("GBWT_B200_DNA_CHECKPOINTS", dna_checkpoints)
    rng = random.Random(300 + seed)
    paths = random_paths(rng, n_nodes=rng.choice([3, 6, 12]), n_paths=rng.choice([10, 40]), max_len=rng.choice([20, 90, 300]))
    if not any(paths):
        paths.append([2, 4])
    b = gb.build_bwt(gb.bidirectional_sequences(paths))
    img = synth.gbwt_image(**image_args(b))
    starts, data = random_labels(rng, (b["alphabet_size"] - (b["offset"] + 1)) // 2, rng.choice([3, 40, 700]))
    gbz = synth.gbz_image(img, starts, data, 4)
    g = orc.GBWT.load(gbz)
    e = index(b200, gbz, monkeypatch, 6)
    dna = dna_of(g)
    check_dna_ranges(e, dna, *dna_ranges(dna, rng))


@pytest.mark.parametrize("dna_checkpoints", ["1", "0"])
def test_dna_bubble_chain(b200, dna_checkpoints, monkeypatch):
    monkeypatch.setenv("GBWT_B200_DNA_CHECKPOINTS", dna_checkpoints)
    S, H, seed = 1500, 8, 11
    img = synth.bubble_chain(S, H, seed)
    starts, data = synth.node_labels(3 * S + 1, seed=5, max_anchor=48)
    gbz = synth.gbz_image(img, starts, data, 4)
    g = orc.GBWT.load(gbz)
    e = index(b200, gbz, monkeypatch, 6)
    dna = dna_of(g)
    rng = random.Random(seed)
    ids, a, b = dna_ranges(dna, rng, 3000)
    check_dna_ranges(e, dna, ids, a, b)
    # a range on the other strand is s ^ 1 at [L - end, L - start), reverse-complemented
    comp = bytes.maketrans(b"ACGTacgtN", b"TGCATGCAN")
    for s in range(0, 2 * H, 2):
        L = len(dna[s])
        x, y = L // 3, L // 3 + 500
        fw = e.extract_dna_ranges([s], [x], [y])[1].tobytes()
        rv = e.extract_dna_ranges([s ^ 1], [L - y], [L - x])[1].tobytes()
        assert rv == fw[::-1].translate(comp)


def test_dna_ranges_need_labels(b200, monkeypatch):
    e = b200.GBWT.from_bytes(open(os.path.join(GOLDEN, "example.gbwt"), "rb").read())
    with pytest.raises(b200.GBWTError) as err:
        e.extract_dna_ranges([0], [0], [3])
    assert err.value.code == b200.E_NO_GRAPH
    lib = b200.library()
    before = b200.kernel_launches()
    assert lib.gbwt_b200_extract_dna_ranges_device(e._h, None, None, None, 0, None, None, None, 0) == b200.E_NO_GRAPH
    assert b200.kernel_launches() == before


# ---- slots, chunks, device calls ---------------------------------------------------------------------------------------

def raw_call(b200, e, dna, ids, starts, ends, offsets, width):
    """The host call into a buffer with a sentinel around and inside the slots."""
    lib = b200.library()
    fn = lib.gbwt_b200_extract_dna_ranges if dna else lib.gbwt_b200_extract_ranges
    buf = np.full(int(offsets[-1]) + 100, SENTINEL, np.uint8) if dna else np.full(int(offsets[-1]) + 100, 2**64 - 2, np.uint64)
    got = np.zeros(len(ids), np.uint64)
    p = lambda a: a.ctypes.data_as(__import__("ctypes").c_void_p)
    rc = fn(e._h, p(ids), p(starts), p(ends), len(ids), p(offsets), p(buf), p(got))
    assert rc == 0, lib.gbwt_b200_last_error().decode()
    return buf, got


@pytest.mark.parametrize("dna", [False, True])
def test_truncated_and_long_slots(b200, dna, monkeypatch):
    S, H, seed = 400, 6, 2
    img = synth.bubble_chain(S, H, seed)
    starts_l, data = synth.node_labels(3 * S + 1, seed=5, max_anchor=40)
    gbz = synth.gbz_image(img, starts_l, data, 4)
    g = orc.GBWT.load(gbz)
    e = index(b200, gbz, monkeypatch, 6)
    full = dna_of(g) if dna else sequences_of(g)
    rng = random.Random(4)
    ids, starts, ends = (dna_ranges if dna else lambda f, r: edge_ranges([len(x) for x in f], 64, r))(full, rng)
    _, want, lengths = sliced(full, ids, starts, ends, np.uint8 if dna else np.uint64)
    want_off = np.zeros(len(ids) + 1, np.uint64)
    np.cumsum(np.where(lengths == U64MAX, 0, lengths), out=want_off[1:])
    sizes = [max(0, int(n) + rng.choice([-3, -1, 0, 0, 2])) if n != U64MAX else rng.choice([0, 2]) for n in lengths]
    offsets = np.zeros(len(ids) + 1, np.uint64)
    offsets[0] = 1000
    np.cumsum(sizes, out=offsets[1:])
    offsets[1:] += 1000
    buf, got = raw_call(b200, e, dna, ids, starts, ends, offsets, 1 if dna else 8)
    assert np.array_equal(got, lengths)
    sentinel = buf[0]
    assert np.all(buf[:1000] == sentinel) and np.all(buf[int(offsets[-1]):] == sentinel)
    for i in range(len(ids)):
        n = 0 if lengths[i] == U64MAX else min(int(lengths[i]), sizes[i])
        assert np.array_equal(buf[int(offsets[i]):int(offsets[i]) + n], want[int(want_off[i]):int(want_off[i]) + n]), i


@pytest.mark.parametrize("budget", [1, 5, 300])
def test_host_chunks(b200, budget, monkeypatch):
    S, H, seed = 300, 6, 8
    img = synth.bubble_chain(S, H, seed)
    starts_l, data = synth.node_labels(3 * S + 1, seed=5, max_anchor=40)
    gbz = synth.gbz_image(img, starts_l, data, 4)
    e = index(b200, gbz, monkeypatch, 6)
    rng = random.Random(budget)
    g = orc.GBWT.load(gbz)
    seqs, dna = sequences_of(g), dna_of(g)
    nodes_q, dna_q = edge_ranges([len(x) for x in seqs], 64, rng, 400), dna_ranges(dna, rng, 400)
    one = (e.extract_ranges(*nodes_q), e.extract_dna_ranges(*dna_q), e.seek(nodes_q[0], nodes_q[1]))
    monkeypatch.setenv("GBWT_B200_HOST_RAGGED_BUDGET", str(budget))
    monkeypatch.setenv("GBWT_B200_HOST_CHUNK_MB", "1")
    before = b200.kernel_launches()
    many = (e.extract_ranges(*nodes_q), e.extract_dna_ranges(*dna_q), e.seek(nodes_q[0], nodes_q[1]))
    assert b200.kernel_launches() - before > (8 if budget < 300 else 0)
    for x, y in zip(one[:2], many[:2]):
        for a, b in zip(x, y):
            assert np.array_equal(a, b)
    assert np.array_equal(one[2], many[2])
    check_node_ranges(e, seqs, *nodes_q)
    check_dna_ranges(e, dna, *dna_q)


def test_device_entry_points(b200, monkeypatch):
    import torch
    from test_gpu_entry_points import dev, filled, host, ptr, run_on, streams
    S, H, seed = 300, 6, 9
    img = synth.bubble_chain(S, H, seed)
    starts_l, data = synth.node_labels(3 * S + 1, seed=5, max_anchor=40)
    gbz = synth.gbz_image(img, starts_l, data, 4)
    e = index(b200, gbz, monkeypatch, 6)
    g = orc.GBWT.load(gbz)
    seqs, dna = sequences_of(g), dna_of(g)
    lib = b200.library()
    rng = random.Random(3)
    for dna_call, full, (ids, a, b) in ((False, seqs, edge_ranges([len(x) for x in seqs], 64, rng, 300)), (True, dna, dna_ranges(dna, rng, 300))):
        width, dtype = (1, np.uint8) if dna_call else (8, np.uint64)
        want_off, want, want_len = sliced(full, ids, a, b, dtype)
        q0 = 7  # a slice of the batch: offsets start above 0
        offsets = want_off + np.uint64(50)
        for stream in streams():
            out = filled((int(offsets[-1]) + 50) * width)
            lengths = filled(8 * len(ids))
            d_ids, d_a, d_b, d_off = dev(ids), dev(a), dev(b), dev(offsets)
            fn = lib.gbwt_b200_extract_dna_ranges_device if dna_call else lib.gbwt_b200_extract_ranges_device
            run_on(b200, stream, lambda s: fn(e._h, ptr(d_ids, 8 * q0), ptr(d_a, 8 * q0), ptr(d_b, 8 * q0), len(ids) - q0,
                                              ptr(d_off, 8 * q0), ptr(out), ptr(lengths, 8 * q0), s))
            got = host(out, dtype)
            lo, hi = int(offsets[q0]), int(offsets[-1])
            assert np.array_equal(got[lo:hi], want[int(want_off[q0]):])
            assert np.all(got[:lo].view(np.uint8) == SENTINEL) and np.all(got[hi:].view(np.uint8) == SENTINEL)
            assert np.array_equal(host(lengths, np.uint64)[q0:], want_len[q0:])
            assert np.all(host(lengths, np.uint8)[:8 * q0] == SENTINEL)
    paths = paths_of(g)
    ids = np.array([s for s, p in enumerate(paths) for _ in range(0, len(p) + 1, 37)], np.uint64)
    idx = np.array([j for p in paths for j in range(0, len(p) + 1, 37)], np.uint64)
    for stream in streams():
        out = filled(16 * len(ids))
        d_ids, d_idx = dev(ids), dev(idx)
        run_on(b200, stream, lambda s: lib.gbwt_b200_seek_device(e._h, ptr(d_ids), ptr(d_idx), len(ids), ptr(out), s))
        assert np.array_equal(host(out, np.uint64).reshape(-1, 2), e.seek(ids, idx).view(np.uint64).reshape(-1, 2))
    torch.cuda.synchronize()


EMPTY_CALLS = {  # every device entry point of gbwt_b200_ranges.h with an empty batch and NULL pointers
    "seek_device": lambda h: (h, None, None, 0, None),
    "extract_ranges_device": lambda h: (h, None, None, None, 0, None, None, None),
    "extract_dna_ranges_device": lambda h: (h, None, None, None, 0, None, None, None),
}


def declared(pattern):
    return set(re.findall(pattern, open(os.path.join(ROOT, "include", "gbwt_b200_ranges.h")).read()))


def test_header_symbols_are_exported(b200):
    names = declared(r"GBWT_B200_API\s+[^;(]*?\b(gbwt_b200_\w+)\s*\(")
    assert len(names) == 6
    lib = b200.library()
    for name in names:
        assert hasattr(lib, name), f"{name} is declared in include/gbwt_b200_ranges.h but not exported"


def test_empty_batches_launch_nothing(b200):
    import torch
    assert declared(r"\bgbwt_b200_(\w+_device)\(") == set(EMPTY_CALLS)
    e = b200.GBWT.load(os.path.join(GOLDEN, "example.gbz"))
    assert e.has_graph()
    lib = b200.library()
    side = torch.cuda.Stream()
    for name, args in EMPTY_CALLS.items():
        for stream in (side.cuda_stream, 0):
            before = b200.kernel_launches()
            assert getattr(lib, "gbwt_b200_" + name)(*args(e._h), stream) == 0, (name, lib.gbwt_b200_last_error().decode())
            assert b200.kernel_launches() == before, name
    torch.cuda.synchronize()


# ---- damaged index, IPC, size ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("checkpoints", [True, False])
def test_invalid_edge_targets(b200, checkpoints, monkeypatch):
    """An edge to a node beyond the alphabet: the walks end there, and the ranges agree with the same handle's extract."""
    edges = [[(1, 0)], [(2, 0), (40, 0)], [(0, 0)]]
    runs = [[(0, 2)], [(1, 1), (0, 1)], [(0, 1)]]
    g0 = orc.GBWT.from_records(edges, runs, sequences=2, size=6, offset=0)
    img = synth.gbwt_image(2, 6, 0, 3, 4, g0.record_starts(), g0.bwt_data())
    monkeypatch.setenv("GBWT_B200_CHECKPOINTS", "1" if checkpoints else "0")
    monkeypatch.setenv("GBWT_B200_CHECKPOINT_SHIFT", "6")
    e = b200.GBWT.from_bytes(img)
    ids = np.arange(e.sequences(), dtype=np.uint64)
    offsets, nodes, lengths = e.extract(ids)
    seqs = [nodes[int(offsets[s]):int(offsets[s + 1])] for s in range(len(ids))]
    rows = [(s, a, b) for s in range(len(ids)) for a in range(4) for b in range(6)]
    q = np.array(rows, np.uint64)
    check_node_ranges(e, seqs, q[:, 0].copy(), q[:, 1].copy(), q[:, 2].copy())
    for s, seq in enumerate(seqs):
        for j in range(len(seq) + 2):
            p = e.seek(s, j)
            assert (p is None) if j >= len(seq) else (p is not None and p.node == seq[j])


def _ipc_child(blob, queries, conn):
    import gbwt_rs_b200 as b200
    try:
        e = b200.GBWT.import_ipc(blob, device=0)
        ids, a, b = queries
        conn.send(("ok", e.extract_ranges(ids, a, b), e.extract_dna_ranges(ids, a, b), e.seek(ids, a)))
    except Exception as exc:  # pragma: no cover
        conn.send(("error", repr(exc)))
    conn.close()


def test_ipc_import_answers_ranges(b200, monkeypatch):
    import multiprocessing as mp
    S, H, seed = 900, 16, 12
    img = synth.bubble_chain(S, H, seed)
    starts_l, data = synth.node_labels(3 * S + 1, seed=5, max_anchor=40)
    e = index(b200, synth.gbz_image(img, starts_l, data, 4), monkeypatch, 6)
    rng = np.random.default_rng(1)
    ids = rng.integers(0, 2 * H, 5000).astype(np.uint64)
    a = rng.integers(0, 3000, 5000).astype(np.uint64)
    b = a + rng.integers(0, 400, 5000).astype(np.uint64)
    want = (e.extract_ranges(ids, a, b), e.extract_dna_ranges(ids, a, b), e.seek(ids, a))
    ctx = mp.get_context("spawn")
    parent, child = ctx.Pipe()
    proc = ctx.Process(target=_ipc_child, args=(e.export_ipc(), (ids, a, b), child))
    proc.start()
    msg = parent.recv()
    proc.join(timeout=60)
    assert msg[0] == "ok", msg
    for w, got in zip(want[:2], msg[1:3]):
        for x, y in zip(w, got):
            assert np.array_equal(x, y)
    assert np.array_equal(want[2], msg[3])


def test_moderate_size(b200, monkeypatch):
    """S = 200 k sites, H = 64 haplotypes, default checkpoints: 2^16 random ranges, and the query patterns of synth.patterns
    (query q is sequence 2h + o at nodes [t, t + 32)) read back as ranges and seeks."""
    S, H, seed = 200_000, 64, 21
    monkeypatch.delenv("GBWT_B200_CHECKPOINTS", raising=False)
    monkeypatch.delenv("GBWT_B200_CHECKPOINT_SHIFT", raising=False)
    img = synth.bubble_chain(S, H, seed)
    e = b200.GBWT.from_bytes(img.array, checkpoints=True)
    g = orc.GBWT.load(img.array)
    n = 1 << 16
    pats = synth.patterns(S, H, seed, n=n, k=32)
    seqs, last = pattern_origins(S, H, n, 32)
    t = last - np.uint64(31)
    off, nodes, lengths = e.extract_ranges(seqs, t, t + np.uint64(32))
    assert np.all(lengths == 32) and np.array_equal(nodes.reshape(n, 32), pats)
    pos = e.seek(seqs, last)
    assert np.array_equal(pos["node"], pats[:, 31])
    rng = np.random.default_rng(seed)
    ids = rng.integers(0, 2 * H, n).astype(np.uint64)
    a = rng.integers(0, 2 * S + 10, n).astype(np.uint64)
    b = a + rng.integers(0, 5000, n).astype(np.uint64)
    few = np.unique(ids)[:8]
    seqs_full = {int(s): np.asarray(g.sequence(int(s)), np.uint64) for s in few}
    keep = np.isin(ids, few)
    _, got, got_len = e.extract_ranges(ids[keep], a[keep], b[keep])
    table = [seqs_full.get(s, np.zeros(0, np.uint64)) for s in range(int(few.max()) + 1)]
    w_off, want, w_len = sliced(table, ids[keep], a[keep], b[keep], np.uint64)
    assert np.array_equal(got, want) and np.array_equal(got_len, w_len)
    # all 2^16 against the same handle's whole-path extraction
    o2, all_nodes, all_len = e.extract(np.arange(2 * H, dtype=np.uint64))
    full = [all_nodes[int(o2[s]):int(o2[s + 1])] for s in range(2 * H)]
    w = sliced(full, ids, a, b, np.uint64)
    for x, y in zip(w, e.extract_ranges(ids, a, b)):
        assert np.array_equal(x, y)
