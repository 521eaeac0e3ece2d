"""locate on the GPU through the C ABI, bit for bit against the oracle's document array (tests/locate_oracle.py): every
position of the fixtures and of random graphs with revisited nodes, the states of every substring of every path, bubble
chains, the 32-bit limits, a record with more than 65 535 samples, flagged against unflagged indexes, device entry
points, an index imported through CUDA IPC, and a damaged index.

Not tested: the GBWT_B200_E_RANGE path for more than 2^32 - 1 samples. It needs an index of 2^32 path nodes at shift 0
(some 64 GB of samples alone), more than a test should allocate."""
import os

import numpy as np
import pytest

import parity_checks as pc
from locate_oracle import NONE, OCCURRENCE, DocumentArray, pattern_origins, states_contain
from oracle import oracle as orc
from synth import synth
from test_limits_layout import U32MAX, bwt_image, far_jump_paths, large_id_shift
from test_oracle_locate import FIXTURES, GOLDEN, random_graph

pytestmark = pytest.mark.gpu

SHIFTS = [0, 1, 3, None]  # None: the default interval (2^10)


@pytest.fixture(scope="module")
def b200():
    import gbwt_rs_b200
    return gbwt_rs_b200


def flagged(b200, image, monkeypatch, shift=None, **kw):
    if shift is None:
        monkeypatch.delenv("GBWT_B200_LOCATE_SHIFT", raising=False)
    else:
        monkeypatch.setenv("GBWT_B200_LOCATE_SHIFT", str(shift))
    return b200.GBWT.from_bytes(image, locate=True, **kw)


def invalid_positions(g, empty_nodes=()):
    rows = [(0, 0), (max(g.first_node() - 1, 0), 0), (g.alphabet_size(), 0), (g.alphabet_size() + 7, 0), (g.first_node(), 2**40),
            (g.first_node(), 2**32)]
    rows += [(v, 0) for v in empty_nodes]
    # one past the end of the first records (i == len)
    rows += [(v, g.record_len(v - g.alphabet_offset())) for v in range(g.first_node(), min(g.alphabet_size(), g.first_node() + 50))
             if g.record_len(v - g.alphabet_offset()) is not None]
    return np.array(rows, orc.POS_DTYPE)


def substring_states(g):
    """The state of every substring of every path (the config-1 enumeration), plus None states."""
    pats = []
    for s in range(g.sequences()):
        p = list(g.sequence(s))
        for i in range(len(p)):
            for j in range(i + 1, min(len(p), i + 8) + 1):
                pats.append(p[i:j])
    states = np.zeros(len(pats) + 3, orc.STATE_DTYPE)
    for q, p in enumerate(pats):
        st = g.find(p[0])
        for v in p[1:]:
            st = g.extend(st, v) if st is not None else None
        if st is not None:
            states[q] = st
    states[-2] = (g.first_node(), 5, 5)  # empty range
    states[-1] = (0, 0, 0)
    return states


def check_positions(e, g, da, extra=None):
    positions = da.positions()
    if extra is not None:
        positions = np.concatenate([positions, extra])
    got = e.locate_positions(positions)
    want = da.locate_batch(positions)
    assert pc.states_equal(got, want)
    return positions


def check_states(e, da, states):
    offsets, occ = e.locate_states(states)
    w_offsets, w_occ = da.locate_states(states)
    assert np.array_equal(offsets, w_offsets) and pc.states_equal(occ, w_occ)
    return offsets, occ


# 1. + 2. fixtures x layouts x shifts: every position, invalid positions, every substring state
@pytest.mark.parametrize("shift", SHIFTS)
@pytest.mark.parametrize("layout", ["auto", "runs"])
@pytest.mark.parametrize("name", FIXTURES)
def test_fixtures(b200, name, layout, shift, monkeypatch):
    raw = open(os.path.join(GOLDEN, name), "rb").read()
    g = orc.GBWT.load(raw)
    da = DocumentArray(g)
    e = flagged(b200, raw, monkeypatch, shift, layout=layout)
    info = e.locate_info()
    assert info["present"] == 1 and info["interval"] == 1 << (10 if shift is None else shift)
    if shift == 0:
        assert info["samples"] == len(da.seq)  # the whole document array
    empty = [v for v in range(g.first_node(), g.alphabet_size()) if g.record_len(v - g.alphabet_offset()) in (None, 0)]
    check_positions(e, g, da, invalid_positions(g, empty))
    states = substring_states(g)
    offsets, occ = check_states(e, da, states)
    # scalar forms
    s0 = states[0]
    assert e.locate(b200.SearchState(int(s0["node"]), range(int(s0["start"]), int(s0["end"])))) == \
        [(int(o["sequence"]), int(o["index"])) for o in occ[int(offsets[0]):int(offsets[1])]]
    assert e.locate(b200.Pos(0, 0)) is None
    # truncated output slots: the first min(count, slot) occurrences of each state, counts in full
    lib = b200.library()
    sizes = np.diff(offsets)
    slots = np.minimum(sizes, np.arange(len(sizes), dtype=np.uint64) % np.uint64(3))
    t_off = np.zeros(len(states) + 1, np.uint64)
    np.cumsum(slots, out=t_off[1:])
    t_occ = np.zeros(int(t_off[-1]), OCCURRENCE)
    counts = np.zeros(len(states), np.uint64)
    e._check(lib.gbwt_b200_locate_states(e._h, b200._ptr(states), len(states), b200._ptr(t_off), b200._ptr(t_occ), b200._ptr(counts)))
    assert np.array_equal(counts, sizes)
    for q in range(len(states)):
        a, b = int(t_off[q]), int(t_off[q + 1])
        assert pc.states_equal(t_occ[a:b], occ[int(offsets[q]):int(offsets[q]) + (b - a)])


# 3. random graphs with revisited nodes, uni- and bidirectional
@pytest.mark.parametrize("shift", [0, 2, None])
@pytest.mark.parametrize("bidirectional", [True, False])
@pytest.mark.parametrize("seed", range(6))
def test_random_graphs(b200, seed, bidirectional, shift, monkeypatch):
    img, _ = random_graph(seed, bidirectional)
    g = orc.GBWT.load(img)
    da = DocumentArray(g)
    e = flagged(b200, img, monkeypatch, shift)
    check_positions(e, g, da, invalid_positions(g))
    check_states(e, da, substring_states(g))


# 4. bubble chains: random positions and the states of synth.patterns
@pytest.mark.parametrize("shift", [3, None])
@pytest.mark.parametrize("model", [dict(), dict(alt_ppm=50_000, tri_mod=4)])
def test_bubble_chains(b200, model, shift, monkeypatch):
    S, H, seed = 3000, 96, 5
    img = synth.bubble_chain(S, H, seed, **model)
    g = orc.GBWT.load(img.array)
    da = DocumentArray(g)
    e = flagged(b200, img.array, monkeypatch, shift)
    rng = np.random.default_rng(shift or 10)
    k = rng.integers(0, len(da.seq), 1_000_000)
    positions = da.positions()[k]
    assert pc.states_equal(e.locate_positions(positions), da.locate_batch(positions))
    n = 20_000
    pats = synth.patterns(S, H, seed, n=n, k=32, **model)
    states = e.find_extend(pats)
    offsets, occ = check_states(e, da, states)
    seqs, idxs = pattern_origins(S, H, n, k=32)
    assert states_contain(offsets, occ, seqs, idxs)


# 5. limits: node ids just below 2^32; a record with more than 65 535 samples
def test_large_node_ids(b200, monkeypatch):
    paths = far_jump_paths()
    shift = large_id_shift(paths)
    img, _ = bwt_image(paths, shift, extra_records=1)
    g = orc.GBWT.load(img)
    assert g.alphabet_size() == U32MAX
    da = DocumentArray(g)
    for s in (0, 4, None):
        e = flagged(b200, img, monkeypatch, s)
        check_positions(e, g, da, invalid_positions(g))
        check_states(e, da, substring_states(g)[:5000])


def test_record_with_many_samples(b200, monkeypatch):
    S, H, seed = 3, 70_000, 9  # 70 000 forward paths through every anchor: at shift 0 its record holds 70 000 samples
    img = synth.bubble_chain(S, H, seed)
    g = orc.GBWT.load(img.array)
    da = DocumentArray(g)
    assert int(np.diff(da.first).max()) > 65_535
    e = flagged(b200, img.array, monkeypatch, 0)
    assert e.locate_info()["samples"] == len(da.seq)
    check_positions(e, g, da)
    states = g.find_batch(np.arange(g.first_node(), g.alphabet_size(), dtype=np.uint64))
    check_states(e, da, states)


# 6. a flagged index answers everything else like an unflagged one; an unflagged index has no samples
def test_flag_changes_nothing_else(b200, monkeypatch):
    S, H, seed = 900, 32, 11
    img = synth.bubble_chain(S, H, seed)
    monkeypatch.delenv("GBWT_B200_LOCATE_SHIFT", raising=False)
    plain, loc = b200.GBWT.from_bytes(img.array), b200.GBWT.from_bytes(img.array, locate=True)
    pats = synth.patterns(S, H, seed, n=30_000, k=32)
    assert pc.states_equal(plain.find_extend(pats), loc.find_extend(pats))
    ids = np.arange(2 * H, dtype=np.uint64)
    for a, b in zip(plain.extract(ids), loc.extract(ids)):
        assert np.array_equal(a, b)
    assert plain.serialize() == loc.serialize()
    info = loc.locate_info()
    assert loc.device_bytes()["total"] == plain.device_bytes()["total"] + info["bytes"]
    assert plain.locate_info()["present"] == 0
    for call in (lambda: plain.locate_positions(np.zeros(1, orc.POS_DTYPE)), lambda: plain.locate_states(np.zeros(1, orc.STATE_DTYPE))):
        with pytest.raises(b200.GBWTError) as err:
            call()
        assert err.value.code == b200.E_NO_SAMPLES
    lib = b200.library()
    assert lib.gbwt_b200_locate_device(plain._h, None, 0, None, None) == b200.E_NO_SAMPLES
    assert lib.gbwt_b200_locate_states_device(plain._h, None, 0, None, None, None, None) == b200.E_NO_SAMPLES
    # the LF-step counter only counts when asked to
    loc.locate_positions(np.array([(int(pats[0, -1]), 0)], orc.POS_DTYPE))
    assert loc.locate_info()["lf_steps"] == 0
    monkeypatch.setenv("GBWT_B200_LOCATE_STATS", "1")
    _, occ = loc.locate_states(plain.find_extend(pats[:100]))
    assert loc.locate_info()["lf_steps"] > 0


# 7. device entry points on a non-default stream
def test_device_entry_points(b200, monkeypatch):
    import torch
    S, H, seed = 900, 32, 11
    img = synth.bubble_chain(S, H, seed)
    g = orc.GBWT.load(img.array)
    da = DocumentArray(g)
    e = flagged(b200, img.array, monkeypatch, 4)
    pats = synth.patterns(S, H, seed, n=5000, k=32)
    states = e.find_extend(pats)
    want_off, want = da.locate_states(states)
    positions = np.ascontiguousarray(da.positions()[::7])
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(stream):
        d_pos = torch.from_numpy(positions.view(np.uint64).astype(np.int64)).to(dev)
        d_occ = torch.empty(2 * len(positions), dtype=torch.int64, device=dev)
        e.locate_device(d_pos.data_ptr(), len(positions), d_occ.data_ptr(), stream.cuda_stream)
        d_states = torch.from_numpy(states.view(np.uint64).astype(np.int64)).to(dev)
        d_offsets = torch.from_numpy(want_off.astype(np.int64)).to(dev)
        d_out = torch.empty(2 * int(want_off[-1]), dtype=torch.int64, device=dev)
        d_counts = torch.empty(len(states), dtype=torch.int64, device=dev)
        e.locate_states_device(d_states.data_ptr(), len(states), d_offsets.data_ptr(), d_out.data_ptr(), d_counts.data_ptr(),
                               stream.cuda_stream)
    stream.synchronize()
    got = d_occ.cpu().numpy().view(np.uint64).view(OCCURRENCE)
    assert pc.states_equal(got, da.locate_batch(positions))
    assert pc.states_equal(d_out.cpu().numpy().view(np.uint64).view(OCCURRENCE), want)
    assert np.array_equal(d_counts.cpu().numpy().view(np.uint64), np.diff(want_off))


# 8. an index exported through IPC and imported by a spawned child answers locate_states identically
def _ipc_child(blob, states, conn):
    import gbwt_rs_b200 as b200
    try:
        e = b200.GBWT.import_ipc(blob, device=0)
        conn.send(("ok", e.locate_states(states), e.locate_info(), e.device_bytes()["total"]))
    except Exception as exc:  # pragma: no cover
        conn.send(("error", repr(exc)))
    conn.close()


def test_ipc_import_answers_locate(b200, monkeypatch):
    import multiprocessing as mp
    S, H, seed = 900, 32, 11
    img = synth.bubble_chain(S, H, seed)
    e = flagged(b200, img.array, monkeypatch, 5)
    states = e.find_extend(synth.patterns(S, H, seed, n=20_000, k=32))
    want = e.locate_states(states)
    ctx = mp.get_context("spawn")
    parent, child = ctx.Pipe()
    proc = ctx.Process(target=_ipc_child, args=(e.export_ipc(), states, child))
    proc.start()
    msg = parent.recv()
    proc.join(timeout=60)
    assert msg[0] == "ok", msg
    (offsets, occ), info, total = msg[1], msg[2], msg[3]
    assert np.array_equal(offsets, want[0]) and pc.states_equal(occ, want[1])
    mine = e.locate_info()
    assert {k: info[k] for k in ("present", "interval", "samples", "bytes")} == {k: mine[k] for k in ("present", "interval", "samples", "bytes")}
    assert total == e.device_bytes()["total"]


# 9. a damaged index (an edge to a node beyond the alphabet) returns, with none where no sample is met
@pytest.mark.parametrize("shift", [0, 5, None])
def test_invalid_edge_targets(b200, shift, monkeypatch):
    edges = [[(1, 0)], [(2, 0), (40, 0)], [(0, 0)]]
    runs = [[(0, 2)], [(1, 1), (0, 1)], [(0, 1)]]
    g0 = orc.GBWT.from_records(edges, runs, sequences=2, size=6, offset=0)
    img = synth.gbwt_image(2, 6, 0, 3, 4, g0.record_starts(), g0.bwt_data())
    g = orc.GBWT.load(img)
    e = flagged(b200, img, monkeypatch, shift)
    positions = np.array([(1, 0), (1, 1), (2, 0), (2, 1), (40, 0), (0, 0), (3, 0)], orc.POS_DTYPE)
    got = e.locate_positions(positions)
    # the walks the oracle can follow: each sequence is (1, x); its positions locate to where its walk put them
    for s in range(2):
        p = g.start(s)
        j = 0
        while p is not None and p[0] < 3:  # (node 40 has no record: no position there)
            row = np.flatnonzero((positions["node"] == p[0]) & (positions["offset"] == p[1]))
            for r in row:
                assert (int(got[r]["sequence"]), int(got[r]["index"])) == (s, j)
            p, j = g.forward(p), j + 1
    assert got[4]["sequence"] == NONE and got[5]["sequence"] == NONE and got[6]["sequence"] == NONE
