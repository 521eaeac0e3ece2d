"""The 16- and 32-bit limits of the device layout and of the window kernels on the GPU, through the C ABI, bit-exact
against the oracle: the indexes of test_limits_layout.py through every kernel family that can meet them (default
dispatch, general kernels, the lean loop with its out-of-line step, forced record windows, 32-bit patterns,
extraction with and without checkpoints and record windows, DNA)."""
import numpy as np
import pytest

import parity_checks as pc
from oracle import oracle as orc
from synth import synth
from test_gpu_window import damaged_batches
from test_limits_layout import (CHAIN_MODEL, CHAIN_SEED, CHAIN_SITES, FAR_SHORTCUT_PATTERNS, LENGTHS, OFFSET_PAIRS,
                                OFFSET_PATTERNS, U32MAX, bwt_image, check_long_record, check_long_record_bd,
                                far_jump_paths, far_shortcut_index, issue_example_index, large_id_shift,
                                long_record_index, long_record_queries, offset_limit_index, offset_limit_queries,
                                row_jump_paths, window_chain)

pytestmark = pytest.mark.gpu

KNOBS = ("FIND_LEAN", "LOCALITY", "FIND_WINDOW", "WINDOW_STATS", "EXTRACT_WINDOW", "EXTRACT_CHECKPOINTS",
         "EXTRACT_WINDOW_THREADS", "CHECKPOINT_SHIFT", "DNA_CHECKPOINTS", "DNA_RELAY", "CKPT_MIN_RUNS", "CKPT_INTERVAL_RUNS")
WINDOWS = dict(LOCALITY=1, FIND_WINDOW=2, WINDOW_STATS=1)   # record windows on any index they can run on
FIND_FAMILIES = [dict(), dict(FIND_LEAN=0), dict(FIND_LEAN=2), dict(FIND_LEAN=3), WINDOWS]


@pytest.fixture(scope="module")
def b200():
    import gbwt_rs_b200
    return gbwt_rs_b200


def knobs(monkeypatch, **values):
    for k in KNOBS:
        if k not in ("CHECKPOINT_SHIFT", "CKPT_MIN_RUNS", "CKPT_INTERVAL_RUNS"):
            monkeypatch.delenv("GBWT_B200_" + k, raising=False)
    for k, v in values.items():
        monkeypatch.setenv("GBWT_B200_" + k, str(v))


def check_find_families(e, g, batches, monkeypatch):
    """find_extend of every batch (u64, and u32 where the nodes fit) under every find/extend kernel family."""
    wants = [g.find_extend_batch(b) for b in batches]
    for family in FIND_FAMILIES:
        knobs(monkeypatch, **family)
        for batch, want in zip(batches, wants):
            assert pc.states_equal(e.find_extend(batch), want), family
            narrow = np.all(batch < 2**32, axis=1)
            if narrow.any():
                assert pc.states_equal(e.find_extend_u32(batch[narrow].astype(np.uint32)), want[narrow]), family
    knobs(monkeypatch)


# ---- A. records of 32-bit length -------------------------------------------------------------------------------------

@pytest.mark.parametrize("config", ["auto", "runs", "runs-checkpoints"])
@pytest.mark.parametrize("length", LENGTHS)
@pytest.mark.parametrize("sigma", [2, 4, 64, 300])
def test_records_of_32_bit_length(b200, sigma, length, config, monkeypatch):
    if config == "runs-checkpoints":
        knobs(monkeypatch, CKPT_MIN_RUNS=1, CKPT_INTERVAL_RUNS=2)
    img = long_record_index(sigma, length)
    g, e = orc.GBWT.load(img), b200.GBWT.from_bytes(img, layout="auto" if config == "auto" else "runs")
    if config == "runs-checkpoints" and sigma <= 64:
        assert e.device_bytes()["records_run_checkpointed"] > 0
    check_long_record(e, g, sigma, length)
    _, _, _, pats2, pats3 = long_record_queries(sigma, length)
    check_find_families(e, g, [pats2, pats3], monkeypatch)


@pytest.mark.parametrize("length", [2**24 + 1, 2**31 + 1, U32MAX])
@pytest.mark.parametrize("sigma", [2, 4, 300])
def test_records_of_32_bit_length_bidirectional(b200, sigma, length, monkeypatch):
    img = long_record_index(sigma, length, bidirectional=True)
    g, e = orc.GBWT.load(img), b200.GBWT.from_bytes(img)
    check_long_record_bd(e, g, sigma)
    knobs(monkeypatch, **WINDOWS)
    check_long_record_bd(e, g, sigma)


@pytest.mark.parametrize("sigma", [2, 300])
def test_record_of_length_2_32_is_rejected(b200, sigma):
    with pytest.raises(b200.GBWTError) as err:
        b200.GBWT.from_bytes(long_record_index(sigma, 2**32))
    assert err.value.code == b200.E_RANGE


# ---- B. edge offset + rank at 2^32 -----------------------------------------------------------------------------------

@pytest.mark.parametrize("layout", ["auto", "runs"])
def test_edge_offset_plus_rank_at_the_limit(b200, layout, monkeypatch):
    img = offset_limit_index()
    g, e = orc.GBWT.load(img), b200.GBWT.from_bytes(img, layout=layout)
    assert int(g.find_extend_batch(OFFSET_PATTERNS)["end"][0]) == U32MAX
    assert int(g.find_extend_batch(OFFSET_PAIRS)["end"][0]) == U32MAX
    check_find_families(e, g, [OFFSET_PATTERNS, OFFSET_PAIRS], monkeypatch)
    states, nodes, pos = offset_limit_queries()
    assert pc.states_equal(e.extend(states, nodes), g.extend_batch(states, nodes))
    assert pc.states_equal(e.forward(pos), g.forward_batch(pos))
    pc.check_find_all_nodes(e, g)


@pytest.mark.parametrize("which", [1, 2, "example"])
def test_edge_offset_plus_rank_over_the_limit_is_rejected(b200, which):
    img = issue_example_index() if which == "example" else offset_limit_index(over=1, which=which)
    for layout in ("auto", "runs"):
        with pytest.raises(b200.GBWTError) as err:
            b200.GBWT.from_bytes(img, layout=layout)
        assert err.value.code == b200.E_RANGE


# ---- C. the 16-bit limits of the window tables -----------------------------------------------------------------------

def bd_random(g, pats, rng):
    n, k = pats.shape
    first = rng.integers(0, k, size=n).astype(np.uint64)
    start = (first * rng.random(n)).astype(np.uint64)
    end = (first + 1 + ((k - first - 1) * rng.random(n)).astype(np.uint64)).astype(np.uint64)
    offs = np.arange(n + 1, dtype=np.uint64) * k
    return pats.reshape(-1), offs, first, start, end


def test_far_shortcut(b200, monkeypatch):
    # the shortcut does not fit the window's 16-bit field: the window takes the two steps one at a time (and defers)
    img = far_shortcut_index()
    g, e = orc.GBWT.load(img), b200.GBWT.from_bytes(img)
    check_find_families(e, g, [FAR_SHORTCUT_PATTERNS], monkeypatch)
    knobs(monkeypatch, **WINDOWS)
    w0 = e.window_info()
    assert pc.states_equal(e.find_extend(FAR_SHORTCUT_PATTERNS), g.find_extend_batch(FAR_SHORTCUT_PATTERNS))
    assert e.window_info()["queries"] > w0["queries"]


@pytest.mark.parametrize("h", [0xFFFE, 0xFFFF, 0x10000, 70000])
def test_window_limit_chains(b200, h, monkeypatch):
    img = window_chain(h)
    g = orc.GBWT.load(img.array)
    knobs(monkeypatch, CHECKPOINT_SHIFT=6, **WINDOWS)
    e = b200.GBWT.from_bytes(img.array, checkpoints=True)
    rng = np.random.default_rng(h)
    w0 = e.window_info()
    assert w0["can_run"]
    for k in (2, 17, 32):
        pats = synth.patterns(CHAIN_SITES, h, CHAIN_SEED, n=20_000, k=k, **CHAIN_MODEL)
        for batch in damaged_batches(g, pats, rng):
            want = g.find_extend_batch(batch)
            assert pc.states_equal(e.find_extend(batch), want), k
            narrow = np.all(batch < 2**32, axis=1)
            assert pc.states_equal(e.find_extend_u32(batch[narrow].astype(np.uint32)), want[narrow]), k
        args = bd_random(g, pats, rng)
        assert pc.states_equal(e.bd_search(*args), g.bd_search_batch(*args))
    w1 = e.window_info()
    assert w1["queries"] > w0["queries"] and 0 < w1["deferred"] - w0["deferred"] < w1["queries"] - w0["queries"], w1
    # ragged batches: suffixes of sampled sequences
    nodes, offsets = [], [0]
    for i in range(0, 2 * h, 1999):
        s = [int(x) for x in synth.sequence(CHAIN_SITES, h, CHAIN_SEED, i, **CHAIN_MODEL)]
        for j in range(0, len(s), 7):
            nodes += s[j:]; offsets.append(len(nodes))
    nodes, offsets = np.array(nodes, dtype=np.uint64), np.array(offsets, dtype=np.uint64)
    assert pc.states_equal(e.find_extend_ragged(nodes, offsets), g.find_extend_ragged(nodes, offsets))
    # follow from a sample of states
    states = g.bd_find_batch(np.arange(g.alphabet_size() + 1, dtype=np.uint64))
    states = states[states["forward"]["end"] > states["forward"]["start"]]
    for backward in (False, True):
        offs, want, counts = g.follow_batch(states, backward=backward)
        got_offs, got, got_counts = e.follow(states, backward)
        assert np.array_equal(got_counts, counts) and np.array_equal(got_offs, offs) and pc.states_equal(got, want)
    # extraction of every sequence, through the record windows and from global memory
    ids = np.arange(2 * h + 1, dtype=np.uint64)
    o_off, o_nodes = g.extract_batch(ids)
    assert np.array_equal(e.sequence_lengths(ids), g.sequence_lengths(ids))
    for window in (2, 0):
        knobs(monkeypatch, EXTRACT_WINDOW=window)
        offsets, nodes, _ = e.extract(ids)
        assert np.array_equal(offsets, o_off) and np.array_equal(nodes, o_nodes), window


# ---- D. node-id distances and large ids ------------------------------------------------------------------------------

LONG_LABELS = (255, 256, 257, 65535, 65536, 70000)


def labelled_image(paths, img, b, seed):
    """A GBZ image of the index with labels of 0-3 bases, and labels of LONG_LABELS bases on nodes of the paths."""
    rng = np.random.default_rng(seed)
    first_id = (b["offset"] + 1) // 2
    n = (b["alphabet_size"] - (b["offset"] + 1)) // 2
    lengths = rng.integers(0, 4, n).astype(np.uint64)
    on_paths = sorted({x >> 1 for p in paths for x in p})
    for j, length in enumerate(LONG_LABELS):
        lengths[on_paths[(7 * j + 3) % len(on_paths)] - first_id] = length
    starts = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(lengths, out=starts[1:])
    data = np.frombuffer(b"ACGTNacgt", dtype=np.uint8)[rng.integers(0, 9, int(starts[-1]))].copy()
    return synth.gbz_image(img, starts, data, 3)


def check_extraction_families(e, g, monkeypatch):
    ids = np.arange(g.sequences() + 2, dtype=np.uint64)
    o_off, o_nodes = g.extract_batch(ids)
    for family in (dict(EXTRACT_WINDOW=2), dict(EXTRACT_WINDOW=0), dict(EXTRACT_CHECKPOINTS=0)):
        knobs(monkeypatch, **family)
        assert np.array_equal(e.sequence_lengths(ids), g.sequence_lengths(ids))
        for _ in range(2):   # (the second time from both ends: the lengths are known)
            offsets, nodes, _ = e.extract(ids)
            assert np.array_equal(offsets, o_off) and np.array_equal(nodes, o_nodes), family
    want_off, want, want_len = g.extract_dna_batch(ids, ord("$"))
    for family in (dict(), dict(DNA_CHECKPOINTS=0), dict(DNA_CHECKPOINTS=0, DNA_RELAY=0)):
        knobs(monkeypatch, **family)
        assert np.array_equal(e.dna_lengths(ids), want_len), family
        offsets, data, lengths = e.extract_dna(ids, ord("$"))
        assert np.array_equal(offsets, want_off) and np.array_equal(lengths, want_len) and np.array_equal(data, want), family
    knobs(monkeypatch)


def check_search_families(e, g, monkeypatch):
    seqs = [p for p in pc.all_sequences(g) if p]
    batches = [np.array(pc.subpath_patterns(seqs, k), dtype=np.uint64) for k in (2, 5, 17)]
    assert e.window_info()["can_run"]   # (forced windows fall back to the general kernels on an index they cannot run on)
    w0 = e.window_info()
    check_find_families(e, g, batches, monkeypatch)
    assert e.window_info()["queries"] - w0["queries"] >= 2 * sum(len(b) for b in batches)   # u64 and u32, through the windows
    args = pc.bd_triples([s[:6] for s in seqs[:: max(1, len(seqs) // 12)]])
    want = g.bd_search_batch(*args)
    for family in (dict(), WINDOWS):
        knobs(monkeypatch, **family)
        assert pc.states_equal(e.bd_search(*args), want)
    knobs(monkeypatch)
    return batches


@pytest.fixture(scope="module")
def far_jumps():
    return far_jump_paths()


@pytest.mark.parametrize("layout", ["auto", "runs"])
def test_far_node_jumps(b200, far_jumps, layout, monkeypatch):
    img, b = bwt_image(far_jumps)
    gbz = labelled_image(far_jumps, img, b, seed=3)
    knobs(monkeypatch, CHECKPOINT_SHIFT=6)
    g, e = orc.GBWT.load(gbz), b200.GBWT.from_bytes(gbz, layout=layout, checkpoints=True)
    assert e.checkpoint_info()["present"] and e.has_graph()
    check_extraction_families(e, g, monkeypatch)
    check_search_families(e, g, monkeypatch)


def test_large_node_ids(b200, far_jumps, monkeypatch):
    shift = large_id_shift(far_jumps)
    img, b = bwt_image(far_jumps, shift, extra_records=1)
    gbz = labelled_image([[x + shift for x in p] for p in far_jumps], img, dict(b, alphabet_size=b["alphabet_size"] + 1), seed=4)
    knobs(monkeypatch, CHECKPOINT_SHIFT=6)
    g, e = orc.GBWT.load(gbz), b200.GBWT.from_bytes(gbz, checkpoints=True)
    assert g.alphabet_size() == U32MAX and e.alphabet_size() == U32MAX and e.alphabet_offset() & (1 << 31)
    check_extraction_families(e, g, monkeypatch)
    batches = check_search_families(e, g, monkeypatch)
    # a real node plus 2^32 at any position: None, never the node it would alias in 32 bits
    pats = batches[1]
    for col in range(pats.shape[1]):
        bad = pats.copy()
        bad[:, col] += np.uint64(2**32)
        want = g.find_extend_batch(bad)
        assert not np.any(want["end"])
        check_find_families(e, g, [bad], monkeypatch)
    # two empty records more: node 2^32 - 1 is in the alphabet, whose size 2^32 is the largest accepted; one more is refused
    img2, _ = bwt_image(far_jumps, shift, extra_records=2)
    g2, e2 = orc.GBWT.load(img2), b200.GBWT.from_bytes(img2)
    assert g2.alphabet_size() == e2.alphabet_size() == 2**32
    nodes = np.array([g2.alphabet_offset() + 1, 2**32 - 3, 2**32 - 2, 2**32 - 1, 2**32, 2**32 + 1], dtype=np.uint64)
    assert pc.states_equal(e2.find(nodes), g2.find_batch(nodes))
    top = pats.copy()
    top[::2, -1] = np.uint64(2**32 - 1)
    check_find_families(e2, g2, [pats, top], monkeypatch)
    with pytest.raises(b200.GBWTError) as err:
        b200.GBWT.from_bytes(bwt_image(far_jumps, shift, extra_records=3)[0])
    assert err.value.code == b200.E_RANGE


@pytest.mark.parametrize("threads", [128, 512])
def test_row_jumps(b200, threads, monkeypatch):
    """Extraction rows across a jump of 0x7FFF .. 0x18000 nodes (test_limits_layout.row_jump_paths): lanes that start
    below the record window step into it from the global layout, and the row must start again where the difference
    leaves the 16-bit range."""
    paths = row_jump_paths()
    img, _ = bwt_image(paths)
    knobs(monkeypatch, CHECKPOINT_SHIFT=6)
    g, e = orc.GBWT.load(img), b200.GBWT.from_bytes(img, checkpoints=True)
    assert e.checkpoint_info()["present"] and e.window_info()["can_run"]
    ids = np.arange(g.sequences() + 2, dtype=np.uint64)
    o_off, o_nodes = g.extract_batch(ids)
    for window in (2, 0):
        knobs(monkeypatch, EXTRACT_WINDOW=window, EXTRACT_WINDOW_THREADS=threads)
        offsets, nodes, _ = e.extract(ids)
        assert np.array_equal(offsets, o_off) and np.array_equal(nodes, o_nodes), window
