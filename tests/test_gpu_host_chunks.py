"""The host entry points across their chunk boundaries, against the oracle and against the same call in one chunk.

Fixed-size calls go through the chunk pipeline of the host entry points (alternating streams, the last chunk cut in
halves); GBWT_B200_HOST_CHUNK_MB=1 makes a batch of 125 000 items take several chunks. Ragged calls (patterns, or
results into caller-given slots) are cut where GBWT_B200_HOST_RAGGED_BUDGET says, and every chunk after the first
reaches its kernels with a non-zero `base`: the first pattern node or output slot of the chunk. The slots here start
well above 0, are exact, truncated, empty or over-long, and belong to ids with and without a result. Each test computes
how many chunks the call must take and checks that at least as many kernels ran."""

import numpy as np
import pytest

import parity_checks as pc
from locate_oracle import OCCURRENCE, DocumentArray
from oracle import oracle as orc
from synth import synth
from test_gpu_entry_points import SENTINEL, bd_search_oracle, bd_triples, check_slots, ragged_batch, slot_offsets
from test_gpu_window import force_windows

pytestmark = pytest.mark.gpu

U64MAX = np.uint64(2**64 - 1)
THREADS = orc.max_threads()
S, H, SEED = 600, 32, 13
N_FIXED = 125_000
BUDGETS = [1, 5, 300]   # one item per chunk; less than one item's result; several items, cut inside a run of empty ones


@pytest.fixture(scope="module")
def b200():
    import gbwt_rs_b200
    return gbwt_rs_b200


@pytest.fixture(scope="module")
def chain():
    """A bubble chain with node labels: the oracle index (with its graph), its document array, the GBZ image."""
    img = synth.bubble_chain(S, H, SEED)
    starts, data = synth.node_labels(3 * S + 1, seed=3, max_anchor=40)
    gbz = synth.gbz_image(img, starts, data, 4)
    g = orc.GBWT.load(gbz)
    return g, DocumentArray(g), gbz


def index(b200, gbz, monkeypatch, **knobs):
    """The chain on the device, created under the given GBWT_B200_* knobs (checkpoints, locate samples)."""
    for k, v in knobs.items():
        monkeypatch.setenv("GBWT_B200_" + k, str(v))
    checkpoints = knobs.get("CHECKPOINTS")
    e = b200.GBWT.from_bytes(gbz, checkpoints=None if checkpoints is None else checkpoints == 1, locate="LOCATE_SHIFT" in knobs)
    for k in knobs:
        monkeypatch.delenv("GBWT_B200_" + k)
    return e


# ---- chunk arithmetic of the library (cabi.cu: chunk_for, run_chunked, ragged_chunk_end) ------------------------------

def fixed_chunks(n, item_bytes, mb=1):
    """(chunks, whether the last chunk was cut in half) of a fixed-size call of n items."""
    chunk = max(1 << 14, (mb << 20) // item_bytes)
    min_items = max(1 << 14, chunk // 16)
    begin, chunks, halved = 0, 0, False
    while begin < n:
        left = n - begin
        count = min(chunk, left)
        if n > chunk and left <= chunk and left // 2 >= min_items:
            count, halved = left // 2, True
        begin, chunks = begin + count, chunks + 1
    return chunks, halved


def ragged_bounds(offsets, item_budget, elem_budget):
    """The first item of every chunk of a ragged call."""
    n, q0, bounds = len(offsets) - 1, 0, []
    offsets = [int(x) for x in offsets]
    while q0 < n:
        bounds.append(q0)
        q1 = min(n, q0 + item_budget)
        if q1 > q0 + 1 and offsets[q1] - offsets[q0] > elem_budget:
            lo, hi = q0 + 1, q1
            while lo < hi:
                mid = lo + (hi - lo + 1) // 2
                if offsets[mid] - offsets[q0] <= elem_budget:
                    lo = mid
                else:
                    hi = mid - 1
            q1 = lo
        q0 = q1
    return bounds


def in_chunks(b200, monkeypatch, knob, value, expected_chunks, call):
    """call() with the knob unset and with knob=value: both results, after checking that the second run launched at
    least one kernel per expected chunk."""
    monkeypatch.delenv(knob, raising=False)
    whole = call()
    monkeypatch.setenv(knob, str(value))
    before = b200.kernel_launches()
    chunked = call()
    assert b200.kernel_launches() - before >= expected_chunks
    monkeypatch.delenv(knob)
    return whole, chunked


def same(a, b):
    if isinstance(a, tuple):
        return all(same(x, y) for x, y in zip(a, b))
    return np.ascontiguousarray(a).tobytes() == np.ascontiguousarray(b).tobytes()


# ---- fixed-size calls --------------------------------------------------------------------------------------------------

FIXED = ["find", "extend_in_place", "bd_find", "extend_forward", "extend_backward", "start", "forward", "backward", "locate",
         "follow_counts", "locate_states_counts", "node_sequence_lengths", "find_extend", "find_extend_u32"]


def fixed_case(name, b200, e, g, da, rng, n):
    """(item bytes of the widest array, call, oracle answer) of one fixed-size host entry point."""
    lib = b200.library()
    lo, hi = max(0, g.alphabet_offset() - 2), g.alphabet_size() + 3
    nodes, nxt = rng.integers(lo, hi, n, dtype=np.uint64), rng.integers(lo, hi, n, dtype=np.uint64)
    live = rng.integers(g.first_node(), g.alphabet_size(), n, dtype=np.uint64)
    pool = np.concatenate([da.positions()[rng.integers(0, len(da.positions()), 3000)],
                           np.array([(0, 0), (g.first_node(), 2**40), (g.alphabet_size() + 5, 0)], orc.POS_DTYPE)])
    positions = pool[rng.integers(0, len(pool), n)]
    if name == "find":
        return 24, lambda: e.find(nodes), g.find_batch(nodes, threads=THREADS)
    if name == "extend_in_place":
        states = g.find_batch(live, threads=THREADS)

        def extend():
            st = states.copy()
            e._check(lib.gbwt_b200_extend(e._h, b200._ptr(st), b200._ptr(nxt), n, b200._ptr(st)))
            return st
        return 24, extend, g.extend_batch(states, nxt, threads=THREADS)
    if name == "bd_find":
        return 48, lambda: e.bd_find(nodes), g.bd_find_batch(nodes, threads=THREADS)
    if name in ("extend_forward", "extend_backward"):
        bd = g.bd_find_batch(live, threads=THREADS)
        backward = name == "extend_backward"
        return 48, lambda: getattr(e, name)(bd, nxt), g.bd_extend_batch(bd, nxt, backward=backward, threads=THREADS)
    if name == "start":
        ids = rng.integers(0, g.sequences() + 5, n, dtype=np.uint64)
        table = np.array([g.start(i) or (0, 0) for i in range(g.sequences() + 5)], orc.POS_DTYPE)
        return 16, lambda: e.start(ids), table[ids]
    if name == "forward":
        return 16, lambda: e.forward(positions), g.forward_batch(positions, threads=THREADS)
    if name == "backward":
        table = np.array([g.backward((int(p["node"]), int(p["offset"]))) or (0, 0) for p in pool], orc.POS_DTYPE)
        pick = rng.integers(0, len(pool), n)
        return 16, lambda: e.backward(pool[pick]), table[pick]
    if name == "locate":
        return 16, lambda: e.locate_positions(positions), da.locate_batch(positions)
    if name == "follow_counts":
        bd = g.bd_find_batch(nodes, threads=THREADS)

        def counts():
            c = np.zeros(n, np.uint64)
            e._check(lib.gbwt_b200_follow(e._h, b200._ptr(bd), n, 0, None, None, b200._ptr(c)))
            return c
        return 48, counts, g.follow_batch(bd, threads=THREADS)[2]
    if name == "locate_states_counts":
        states = g.find_batch(nodes, threads=THREADS)

        def counts():
            c = np.zeros(n, np.uint64)
            e._check(lib.gbwt_b200_locate_states(e._h, b200._ptr(states), n, None, None, b200._ptr(c)))
            return c
        return 24, counts, np.where(states["end"] > states["start"], states["end"] - states["start"], 0).astype(np.uint64)
    if name == "node_sequence_lengths":
        top = g.alphabet_size() // 2 + 5
        table = np.array([len(x) if x is not None else U64MAX for x in (g.node_sequence(i) for i in range(top))], np.uint64)
        ids = rng.integers(0, top, n, dtype=np.uint64)
        return 16, lambda: e.node_sequence_lengths(ids), table[ids]
    k = 8
    pats = synth.patterns(S, H, SEED, n=n, k=k)
    pats[::5, 3] ^= np.uint64(1)
    want = g.find_extend_batch(pats, threads=THREADS)
    if name == "find_extend":
        return 8 * k, lambda: e.find_extend(pats), want
    return 4 * k, lambda: e.find_extend_u32(pats.astype(np.uint32)), want


@pytest.mark.parametrize("name", FIXED)
def test_fixed_size_calls_across_chunks(b200, chain, name, monkeypatch):
    g, da, gbz = chain
    e = index(b200, gbz, monkeypatch, LOCATE_SHIFT=3)
    item_bytes, call, want = fixed_case(name, b200, e, g, da, np.random.default_rng(FIXED.index(name)), N_FIXED)
    chunks, halved = fixed_chunks(N_FIXED, item_bytes)
    assert chunks >= 3 and (halved or item_bytes != 24)   # two full chunks at least, and a halved tail for 24-byte items
    whole, chunked = in_chunks(b200, monkeypatch, "GBWT_B200_HOST_CHUNK_MB", 1, chunks, call)
    assert same(whole, want) and same(chunked, want)


# ---- ragged inputs -----------------------------------------------------------------------------------------------------

def ragged_patterns(g, rng, n=3000):
    pats = synth.patterns(S, H, SEED, n=n, k=24, seed_q=5)
    pats[::7, 5] ^= np.uint64(1)
    return ragged_batch(pats, rng, prefix=11)


@pytest.mark.parametrize("budget", BUDGETS)
def test_find_extend_ragged_across_chunks(b200, chain, budget, monkeypatch):
    g, _, gbz = chain
    e = index(b200, gbz, monkeypatch)
    nodes, offsets = ragged_patterns(g, np.random.default_rng(budget))
    want = g.find_extend_ragged(nodes, offsets, threads=THREADS)
    bounds = ragged_bounds(offsets, min(1 << 20, budget), min(8 << 20, budget))
    whole, chunked = in_chunks(b200, monkeypatch, "GBWT_B200_HOST_RAGGED_BUDGET", budget, len(bounds),
                               lambda: e.find_extend_ragged(nodes, offsets))
    assert pc.states_equal(whole, want) and pc.states_equal(chunked, want)
    assert np.count_nonzero(want["end"] > want["start"]) > len(want) // 4


@pytest.mark.parametrize("direct", ["1", "0"])
@pytest.mark.parametrize("windows", [True, False])
@pytest.mark.parametrize("budget", BUDGETS)
def test_bd_search_across_chunks(b200, chain, budget, windows, direct, monkeypatch):
    g, _, gbz = chain
    e = index(b200, gbz, monkeypatch)
    if windows:
        force_windows(monkeypatch)
    monkeypatch.setenv("GBWT_B200_WINDOW_DIRECT", direct)
    rng = np.random.default_rng(10 + budget)
    nodes, offsets = ragged_patterns(g, rng)
    first, start, end = bd_triples(offsets, rng)
    want = bd_search_oracle(g, nodes, offsets, first, start, end)
    bounds = ragged_bounds(offsets, min(1 << 20, budget), min(8 << 20, budget))
    whole, chunked = in_chunks(b200, monkeypatch, "GBWT_B200_HOST_RAGGED_BUDGET", budget, len(bounds),
                               lambda: e.bd_search(nodes, offsets, first, start, end))
    assert pc.states_equal(whole, want) and pc.states_equal(chunked, want)
    assert np.count_nonzero(want["forward"]["end"] > want["forward"]["start"]) > len(want) // 4
    if windows:
        # the record windows took the chunks: with them turned off (GBWT_B200_BD_WINDOW=0, the general kernel after the
        # same sort) the same call launches a different number of kernels, and answers the same
        monkeypatch.setenv("GBWT_B200_HOST_RAGGED_BUDGET", str(budget))
        launches = []
        for bd_window in ("1", "0"):
            monkeypatch.setenv("GBWT_B200_BD_WINDOW", bd_window)
            before = b200.kernel_launches()
            assert pc.states_equal(e.bd_search(nodes, offsets, first, start, end), want)
            launches.append(b200.kernel_launches() - before)
        assert launches[0] != launches[1], launches


# ---- results into slots ------------------------------------------------------------------------------------------------

def into_slots(b200, e, fn, items, offsets, dtype, mid=()):
    """fn(index, items, n, *mid, out_offsets, out, lengths) into a sentinel-filled buffer: (out bytes, lengths)."""
    w = np.dtype(dtype).itemsize
    out = np.full((int(offsets[-1]) + 20) * w, SENTINEL, np.uint8)
    lengths = np.full(len(items), 7, np.uint64)
    e._check(fn(e._h, b200._ptr(items), len(items), *mid, b200._ptr(offsets), b200._ptr(out), b200._ptr(lengths)))
    return out, lengths


def check_slot_call(b200, e, monkeypatch, budget, fn, items, sizes, want_lengths, truth, dtype, mid=(), item_budget=None,
                    elem_budget=None):
    """A slot-writing host call with budget `budget`, slots from 1000 on: lengths in full, result i cut to slot i, nothing
    written outside the slots; the same bytes in the slots as with one chunk; enough kernels for the chunks."""
    offsets = slot_offsets(sizes, first=1000)
    bounds = ragged_bounds(offsets, min(item_budget or len(items), budget), min(elem_budget or 2**62, budget))
    assert len(bounds) > 1
    run = len(items) // 3   # (slot_offsets makes slots run .. run + 8 empty)
    assert budget > 8 or any(run < b < run + 8 for b in bounds)
    whole, chunked = in_chunks(b200, monkeypatch, "GBWT_B200_HOST_RAGGED_BUDGET", budget, len(bounds),
                               lambda: into_slots(b200, e, fn, items, offsets, dtype, mid))
    for out, lengths in (whole, chunked):
        assert np.array_equal(lengths, want_lengths)
        check_slots(out, dtype, offsets, truth)
    w = np.dtype(dtype).itemsize
    for i in range(len(items)):   # what a slot holds beyond its result is unspecified; the result is not
        a = int(offsets[i]) * w
        m = min(int(offsets[i + 1] - offsets[i]), int(sizes[i])) * w
        assert whole[0][a:a + m].tobytes() == chunked[0][a:a + m].tobytes(), i


@pytest.mark.parametrize("backward", [0, 1])
@pytest.mark.parametrize("budget", BUDGETS)
def test_follow_into_slots(b200, chain, budget, backward, monkeypatch):
    g, _, gbz = chain
    e = index(b200, gbz, monkeypatch)
    rng = np.random.default_rng(budget)
    states = g.bd_find_batch(np.arange(g.alphabet_size() + 3, dtype=np.uint64), threads=THREADS)
    states = np.concatenate([states, g.bd_extend_batch(states[rng.integers(0, len(states), 600)],
                                                       rng.integers(0, g.alphabet_size(), 600, dtype=np.uint64), backward=bool(backward))])
    w_off, want, counts = g.follow_batch(states, backward=bool(backward), threads=THREADS)
    sizes = np.where(counts == U64MAX, np.uint64(0), counts)
    check_slot_call(b200, e, monkeypatch, budget, b200.library().gbwt_b200_follow, states, sizes, counts,
                    lambda i: want[int(w_off[i]):int(w_off[i + 1])], orc.BDSTATE_DTYPE, mid=(backward,),
                    item_budget=1 << 20, elem_budget=4 << 20)


@pytest.mark.parametrize("budget", BUDGETS)
def test_locate_states_into_slots(b200, chain, budget, monkeypatch):
    g, da, gbz = chain
    e = index(b200, gbz, monkeypatch, LOCATE_SHIFT=2)
    pats = synth.patterns(S, H, SEED, n=900, k=3, seed_q=9)
    pats[::4, 1] ^= np.uint64(1)
    states = np.concatenate([g.find_extend_batch(pats, threads=THREADS), g.find_batch(np.arange(g.alphabet_size() + 2, dtype=np.uint64))])
    w_off, w_occ = da.locate_states(states)
    sizes = np.diff(w_off)
    check_slot_call(b200, e, monkeypatch, budget, b200.library().gbwt_b200_locate_states, states, sizes, sizes,
                    lambda i: w_occ[int(w_off[i]):int(w_off[i + 1])], OCCURRENCE, item_budget=1 << 22, elem_budget=16 << 20)


@pytest.mark.parametrize("budget", BUDGETS)
def test_node_sequences_into_slots(b200, chain, budget, monkeypatch):
    g, _, gbz = chain
    e = index(b200, gbz, monkeypatch)
    top = g.alphabet_size() // 2 + 4
    rng = np.random.default_rng(budget)
    ids = rng.permutation(np.concatenate([rng.permutation(top)[:700], [0, top - 1, 2**40]]).astype(np.uint64))
    labels = [g.node_sequence(int(i)) for i in ids]
    want_lengths = np.array([len(x) if x is not None else U64MAX for x in labels], np.uint64)
    assert np.any(want_lengths == U64MAX)
    check_slot_call(b200, e, monkeypatch, budget, b200.library().gbwt_b200_node_sequences, ids,
                    np.where(want_lengths == U64MAX, np.uint64(0), want_lengths), want_lengths,
                    lambda i: np.frombuffer(labels[i] or b"", np.uint8), np.uint8)


def sequence_ids(g, rng, copies=2):
    ids = np.concatenate([np.arange(g.sequences(), dtype=np.uint64),
                          np.array([g.sequences(), g.sequences() + 1, 2**40], dtype=np.uint64)])
    return rng.permutation(np.tile(ids, copies))


# GBWT_B200_* knobs of each extraction family: at index creation, and at the call
EXTRACT = {
    "checkpointed": (dict(CHECKPOINTS=1, CHECKPOINT_SHIFT=6), dict(EXTRACT_WINDOW=0)),
    "checkpointed-windows": (dict(CHECKPOINTS=1, CHECKPOINT_SHIFT=6), dict(EXTRACT_WINDOW=2)),
    "two-ended": (dict(CHECKPOINTS=0), dict()),
    "one-ended": (dict(CHECKPOINTS=0), dict(EXTRACT_SPLIT=0)),
    "lanes-1": (dict(CHECKPOINTS=0), dict(EXTRACT_STRIDE=1)),
    "lanes-4": (dict(CHECKPOINTS=1, CHECKPOINT_SHIFT=6), dict(EXTRACT_STRIDE=4)),
}


def check_extract(b200, e, g, budget, rng, monkeypatch, measured, copies=2):
    ids = sequence_ids(g, rng, copies)
    o_off, o_nodes = g.extract_batch(ids, threads=THREADS)
    lengths = g.sequence_lengths(ids, threads=THREADS)
    if measured:   # lengths known: the two-ended walks
        assert np.array_equal(e.sequence_lengths(ids), lengths)
    check_slot_call(b200, e, monkeypatch, budget, b200.library().gbwt_b200_extract, ids, np.diff(o_off), lengths,
                    lambda i: o_nodes[int(o_off[i]):int(o_off[i + 1])], np.uint64)


@pytest.mark.parametrize("family", list(EXTRACT))
@pytest.mark.parametrize("budget", BUDGETS)
def test_extract_into_slots(b200, chain, budget, family, monkeypatch):
    g, _, gbz = chain
    created, called = EXTRACT[family]
    e = index(b200, gbz, monkeypatch, **created)
    assert e.checkpoint_info()["present"] == created["CHECKPOINTS"]
    for k, v in called.items():
        monkeypatch.setenv("GBWT_B200_" + k, str(v))
    check_extract(b200, e, g, budget, np.random.default_rng(budget), monkeypatch, measured=family == "two-ended")


@pytest.mark.parametrize("checkpoints", [True, False])
@pytest.mark.parametrize("budget", BUDGETS)
def test_checked_extract_into_slots(b200, budget, checkpoints, monkeypatch):
    # an edge to a node beyond the alphabet: the bounds-checked kernels (see test_checkpoints_on_an_index_with_invalid_edge_targets)
    edges = [[(1, 0)], [(2, 0), (40, 0)], [(0, 0)]]
    runs = [[(0, 2)], [(1, 1), (0, 1)], [(0, 1)]]
    g0 = orc.GBWT.from_records(edges, runs, sequences=2, size=6, offset=0)
    img = synth.gbwt_image(2, 6, 0, 3, 4, g0.record_starts(), g0.bwt_data())
    g, e = orc.GBWT.load(img), b200.GBWT.from_bytes(img, checkpoints=checkpoints)
    assert e.checkpoint_info()["present"] == checkpoints
    check_extract(b200, e, g, budget, np.random.default_rng(budget), monkeypatch, measured=not checkpoints, copies=100)


DNA = {
    "checkpointed": (dict(CHECKPOINTS=1, CHECKPOINT_SHIFT=6), dict()),
    "relay": (dict(CHECKPOINTS=0), dict()),
    "split": (dict(CHECKPOINTS=0), dict(DNA_RELAY=0)),
    "whole-walks": (dict(CHECKPOINTS=1, CHECKPOINT_SHIFT=6), dict(DNA_CHECKPOINTS=0, EXTRACT_SPLIT=0)),
}


@pytest.mark.parametrize("family", list(DNA))
@pytest.mark.parametrize("budget", BUDGETS)
def test_extract_dna_into_slots(b200, chain, budget, family, monkeypatch):
    g, _, gbz = chain
    created, called = DNA[family]
    e = index(b200, gbz, monkeypatch, **created)
    for k, v in called.items():
        monkeypatch.setenv("GBWT_B200_" + k, str(v))
    ids = sequence_ids(g, np.random.default_rng(budget))
    endmarker = ord("$")
    w_off, w_bytes, lengths = g.extract_dna_batch(ids, endmarker, threads=THREADS)
    assert np.array_equal(e.dna_lengths(ids), lengths)   # (measured: the relay and split kernels spell from both ends)
    check_slot_call(b200, e, monkeypatch, budget, b200.library().gbwt_b200_extract_dna, ids, np.diff(w_off), lengths,
                    lambda i: w_bytes[int(w_off[i]):int(w_off[i + 1])], np.uint8, mid=(endmarker,))
