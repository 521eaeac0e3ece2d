"""The 16- and 32-bit limits of the device layout, checked on the CPU (tests/hostsim: the product's layout builder and
record_scan.cuh) against the oracle. The layout narrows what the reference keeps as usize: record lengths, edge
offsets and node ids are u32, the record-window tables of find_window.cu use 16-bit fields. Every construction here
sits on one of those limits, and every test asserts from the descriptors that it really does. The same indexes go
through the GPU kernels in test_gpu_limits.py."""
import random

import numpy as np
import pytest

import gbwt_builder as gb
import parity_checks as pc
from hostsim_build import HostSim
from oracle import oracle as orc
from synth import synth
from test_hostsim_layout import records_image

U32MAX = 2**32 - 1
FMT_SINGLE, FMT_DENSE2, FMT_RUN32, FMT_RUN64 = 1, 2, 4, 5
LENGTHS = [2**24 - 1, 2**24, 2**24 + 1, 2**31 - 1, 2**31, 2**31 + 1, U32MAX]


def desc(e, rec):
    """(total_len, fmt, checkpoint shift or None, body_len, w01, w23) of one descriptor (layout.h: RecordDesc)."""
    w = [int(x) for x in e.desc_words(rec)]
    ckpt = (w[1] >> 25) & 31
    return w[0], (w[1] >> 16) & 0xFF, (ckpt - 1 if ckpt else None), w[5], (w[2], w[3]), (w[6], w[7])


# ---- A. records of 32-bit length -------------------------------------------------------------------------------------

def long_record_index(sigma, length, bidirectional=False):
    """Record 1 has `sigma` successors (nodes 2 .. sigma + 1) and `length` positions in a handful of runs, so it costs
    bytes, not gigabytes; with more than four symbols, one run of length 1 per symbol comes first. Run boundaries lie
    at 2^24 +- 1 and around the middle. Successor v is a single-edge record back to the endmarker."""
    runs = [(v, 1) for v in range(sigma)] if sigma > 4 else []
    pos = len(runs)
    bounds = sorted(b for b in {1, 2**24 - 1, 2**24 + 1, length // 2 + 3, length - 1} if pos < b < length) + [length]
    for j, b in enumerate(bounds):
        runs.append((j % min(sigma, 4), b - pos))
        pos = b
    counts = [0] * sigma
    for v, n in runs:
        counts[v] += n
    edges = [[(1, 0)], [(2 + v, 0) for v in range(sigma)]] + [[(0, 0)] for _ in range(sigma)]
    rr = [[(0, 3)], runs] + [[(0, max(1, c))] for c in counts]
    img, _ = records_image(edges, rr, sequences=3, size=3, offset=0, bidirectional=bidirectional)
    return img


def cuts(length):
    return sorted({0, 1, 2**24 - 1, 2**24 + 1, 2**31 - 1, 2**31 + 1, length - 1, length, length + 1, 2**40})


def probe_nodes(sigma):
    """Every successor of the long record for small sigma, a sample for wide records, and nodes that are none."""
    succ = list(range(2, 2 + sigma)) if sigma <= 4 else [2, 3, 4, 5, sigma // 2 + 2, sigma + 1]
    return sorted(set(succ + [0, 1, sigma + 2, sigma + 9, 2**32 + 2, 2**33]))


def long_record_queries(sigma, length):
    st, nx = [], []
    cc = cuts(length)
    for a in cc:
        for b in cc:
            if a < b:
                for node in probe_nodes(sigma):
                    st.append((1, a, b)); nx.append(node)
    states = np.array(st, dtype=orc.STATE_DTYPE)
    nodes = np.array(nx, dtype=np.uint64)
    pos = np.array([(1, c) for c in cc] + [(2, c) for c in cc] + [(sigma + 1, c) for c in cc], dtype=orc.POS_DTYPE)
    pats2 = np.array([[1, n] for n in probe_nodes(sigma)] + [[n, 0] for n in probe_nodes(sigma)], dtype=np.uint64)
    pats3 = np.array([[1, n, 0] for n in probe_nodes(sigma)] + [[0, 1, n] for n in probe_nodes(sigma)], dtype=np.uint64)
    return states, nodes, pos, pats2, pats3


def check_long_record(e, g, sigma, length):
    states, nodes, pos, pats2, pats3 = long_record_queries(sigma, length)
    want = g.extend_batch(states, nodes)
    assert pc.states_equal(e.extend(states, nodes), want)
    assert int(want["end"].max()) >= length // 4   # (the largest symbol holds at least a quarter of the record)
    assert pc.states_equal(e.forward(pos), g.forward_batch(pos))
    pc.check_find_all_nodes(e, g)
    for pats in (pats2, pats3):
        assert pc.states_equal(e.find_extend(pats), g.find_extend_batch(pats))
    flat = np.concatenate([pats2.reshape(-1), pats3.reshape(-1)])
    offsets = np.array([0] + [2 * (i + 1) for i in range(len(pats2))] + [2 * len(pats2) + 3 * (i + 1) for i in range(len(pats3))],
                       dtype=np.uint64)
    assert pc.states_equal(e.find_extend_ragged(flat, offsets), g.find_extend_ragged(flat, offsets))


def check_long_record_bd(e, g, sigma):
    nodes = np.arange(g.alphabet_size() + 2, dtype=np.uint64)
    states = g.bd_find_batch(nodes)
    assert pc.states_equal(e.bd_find(nodes), states)
    live = states[states["forward"]["end"] > states["forward"]["start"]]
    probe = np.array(probe_nodes(sigma), dtype=np.uint64)
    rep, nxt = np.repeat(live, len(probe)), np.tile(probe, len(live))
    assert pc.states_equal(e.extend_forward(rep, nxt), g.bd_extend_batch(rep, nxt, backward=False))
    assert pc.states_equal(e.extend_backward(rep, nxt), g.bd_extend_batch(rep, nxt, backward=True))
    args = pc.bd_triples([[1, int(n)] for n in probe if 2 <= n < sigma + 2])
    assert pc.states_equal(e.bd_search(*args), g.bd_search_batch(*args))


def assert_long_layout(e, sigma, length, forced_checkpoints):
    total, fmt, shift, body_len, _, _ = desc(e, 1)
    assert total == length
    assert fmt == (FMT_RUN64 if sigma > 256 else FMT_RUN32)
    if fmt == FMT_RUN32:
        assert body_len >= -(-length // 2**24)   # runs split at 2^24 positions
    if sigma > 64:
        assert shift is None
    elif forced_checkpoints:
        assert shift is not None
    if shift is not None:
        assert (length - 1) >> shift >= 1


@pytest.fixture
def forced(monkeypatch):
    monkeypatch.setenv("GBWT_B200_CKPT_MIN_RUNS", "1")
    monkeypatch.setenv("GBWT_B200_CKPT_INTERVAL_RUNS", "2")


@pytest.mark.parametrize("checkpoints", [False, True])
@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("length", LENGTHS)
@pytest.mark.parametrize("sigma", [2, 3, 4, 64, 300])
def test_records_of_32_bit_length(sigma, length, layout, checkpoints, request):
    if checkpoints:
        request.getfixturevalue("forced")
    img = long_record_index(sigma, length)
    g, e = orc.GBWT.load(img), HostSim(img, layout)
    assert_long_layout(e, sigma, length, checkpoints)
    check_long_record(e, g, sigma, length)


@pytest.mark.parametrize("length", [2**24 + 1, 2**31 + 1, U32MAX])
@pytest.mark.parametrize("sigma", [2, 4, 300])
def test_records_of_32_bit_length_bidirectional(sigma, length):
    img = long_record_index(sigma, length, bidirectional=True)
    g, e = orc.GBWT.load(img), HostSim(img)
    assert g.is_bidirectional()
    check_long_record_bd(e, g, sigma)


def test_checkpoint_shift_reaches_its_cap(forced):
    # 64 symbols over 2^32 - 1 positions: the table doubles P up to 2^30, so entries hold j << 30 up to 3 << 30
    img = long_record_index(64, U32MAX)
    e = HostSim(img, 1)
    assert desc(e, 1)[2] == 30
    check_long_record(e, orc.GBWT.load(img), 64, U32MAX)


@pytest.mark.parametrize("sigma", [1, 2, 3, 300])
def test_record_of_length_2_32_is_rejected(sigma):
    if sigma == 1:
        edges, rr = [[(1, 0)], [(0, 0)]], [[(0, 3)], [(0, 2**31), (0, 2**31)]]
        img, _ = records_image(edges, rr, sequences=3, size=3, offset=0)
    else:
        img = long_record_index(sigma, 2**32)
    assert orc.GBWT.load(img).record_len(1) == 2**32   # the reference loads it
    with pytest.raises(IOError, match="32-bit"):
        HostSim(img)


# ---- B. edge offset + rank at 2^32 -----------------------------------------------------------------------------------

def offset_limit_index(over=0, which=2):
    """Record 1: edges to nodes 2 and 3, length 2^32 - 1, four runs. Record 2: one edge to node 4, length 2^31 + 2^24.
    The offset of record 2's edge (which=2) or of record 1's edge to node 3 (which=1) is chosen so that
    offset_b + count_b = 2^32 - 1 + over. over = 0 is the largest index the device layout holds."""
    c0 = 2**31 + 2**24                       # positions of record 1 with symbol 0 = length of record 2
    c1 = U32MAX - c0
    runs1 = [(0, 2**24 + 5), (1, 2**20), (0, c0 - 2**24 - 5), (1, c1 - 2**20)]
    off2 = U32MAX - c0 + (over if which == 2 else 0)
    off3 = U32MAX - c1 + (over if which == 1 else 0)
    edges = [[(1, 0)], [(2, 0), (3, off3)], [(4, off2)], [(0, 0)], [(0, 0)]]
    runs = [[(0, 3)], runs1, [(0, c0)], [(0, c1)], [(0, U32MAX)]]
    img, _ = records_image(edges, runs, sequences=3, size=3, offset=0)
    return img


def issue_example_index():
    """The over-limit index that the 32-bit find loops would wrap on: record 2's edge to node 4 has offset
    2^32 - 100 and carries 2^31 + 2^24 positions, so its answers reach end = 0x180FFFF9C."""
    c0 = 2**31 + 2**24
    runs1 = [(0, 2**24 + 5), (1, 2**20), (0, c0 - 2**24 - 5), (1, U32MAX - c0 - 2**20)]
    edges = [[(1, 0)], [(2, 0), (3, 0)], [(4, 2**32 - 100)], [(0, 0)], [(0, 0)]]
    runs = [[(0, 3)], runs1, [(0, c0)], [(0, U32MAX - c0)], [(0, 2**31)]]
    img, _ = records_image(edges, runs, sequences=3, size=3, offset=0)
    return img


OFFSET_PATTERNS = np.array([[1, 2, 4], [1, 3, 4], [2, 4, 0], [1, 2, 3], [0, 1, 2]], dtype=np.uint64)
OFFSET_PAIRS = np.array([[1, 3], [1, 2], [2, 4], [3, 0], [0, 1]], dtype=np.uint64)


def offset_limit_queries():
    cc = sorted({0, 1, 2**24 + 4, 2**24 + 5, 2**24 + 6, 2**31, 2**31 + 2**24 - 1, 2**31 + 2**24, U32MAX - 1, U32MAX, 2**32})
    st, nx = [], []
    for rec in (1, 2):
        for a in cc:
            for b in cc:
                if a < b:
                    for node in (2, 3, 4, 0, 5):
                        st.append((rec, a, b)); nx.append(node)
    pos = np.array([(r, c) for r in (1, 2, 3) for c in cc], dtype=orc.POS_DTYPE)
    return np.array(st, dtype=orc.STATE_DTYPE), np.array(nx, dtype=np.uint64), pos


@pytest.mark.parametrize("layout", [0, 1])
def test_edge_offset_plus_rank_at_the_limit(layout):
    img = offset_limit_index()
    g, e = orc.GBWT.load(img), HostSim(img, layout)
    assert desc(e, 2)[1] == FMT_SINGLE and desc(e, 2)[4][1] == U32MAX - (2**31 + 2**24)
    want = g.find_extend_batch(OFFSET_PATTERNS)
    pairs = g.find_extend_batch(OFFSET_PAIRS)
    assert int(want["end"][0]) == U32MAX and int(pairs["end"][0]) == U32MAX   # over the single edge and over the run body
    assert pc.states_equal(e.find_extend(OFFSET_PATTERNS), want)
    assert pc.states_equal(e.find_extend(OFFSET_PAIRS), pairs)
    states, nodes, pos = offset_limit_queries()
    assert pc.states_equal(e.extend(states, nodes), g.extend_batch(states, nodes))
    assert pc.states_equal(e.forward(pos), g.forward_batch(pos))
    pc.check_find_all_nodes(e, g)


@pytest.mark.parametrize("which", [1, 2])
def test_edge_offset_plus_rank_over_the_limit_is_rejected(which):
    img = offset_limit_index(over=1, which=which)
    g = orc.GBWT.load(img)
    # the reference answers past 2^32 - 1: an index the 32-bit kernels cannot hold
    want = g.find_extend_batch(OFFSET_PATTERNS[:1]) if which == 2 else g.find_extend_batch(OFFSET_PAIRS[:1])
    assert int(want["end"][0]) == 2**32
    for layout in (0, 1):
        with pytest.raises(IOError, match="32-bit"):
            HostSim(img, layout)


def test_issue_example_is_rejected():
    img = issue_example_index()
    g = orc.GBWT.load(img)
    assert tuple(int(x) for x in g.find_extend_batch(OFFSET_PATTERNS[:1])[0]) == (4, 0xFFFFFF9C, 0x180FFFF9C)
    with pytest.raises(IOError, match="32-bit"):
        HostSim(img)


# ---- C. the 16-bit limits of the window tables -----------------------------------------------------------------------

def far_shortcut_index():
    """Records 1 -> 2 -> 3, each with one edge: the two-hop shortcut of record 1 lands on record 3 at offset 0x10000, which
    the 16-bit shortcut field of a record window cannot hold. Record 3 is longer than 0xFFFF, so it is never staged."""
    edges = [[(1, 0)], [(2, 0)], [(3, 0x10000)], [(0, 0)]]
    runs = [[(0, 3)], [(0, 3)], [(0, 3)], [(0, 0x10003)]]
    img, _ = records_image(edges, runs, sequences=3, size=3, offset=0)
    return img


FAR_SHORTCUT_PATTERNS = np.array([[1, 2, 3], [2, 3, 0], [0, 1, 2], [1, 2, 2]], dtype=np.uint64)


def test_far_shortcut():
    img = far_shortcut_index()
    g, e = orc.GBWT.load(img), HostSim(img)
    assert [int(x) for x in e.skips()[1]] == [3, 0x10000, 0, 0]
    want = g.find_extend_batch(FAR_SHORTCUT_PATTERNS)
    assert tuple(int(x) for x in want[0]) == (3, 0x10000, 0x10003)
    assert pc.states_equal(e.find_extend(FAR_SHORTCUT_PATTERNS), want)


CHAIN_SITES, CHAIN_SEED = 40, 3
CHAIN_MODEL = dict(alt_ppm=50_000, tri_mod=5)


def window_chain(h):
    return synth.bubble_chain(CHAIN_SITES, h, CHAIN_SEED, **CHAIN_MODEL)


def window_limits(e):
    """(longest record but the endmarker, records shorter than 0xFFFF with an inline edge offset above 0xFFFF)."""
    longest, far = 0, 0
    for rec in range(1, e.records()):
        total, fmt, _, _, w01, w23 = desc(e, rec)
        longest = max(longest, total)
        if fmt in (FMT_SINGLE, FMT_DENSE2) and total < 0xFFFF and max(w01[1], w23[1] if fmt == FMT_DENSE2 else 0) > 0xFFFF:
            far += 1
    return longest, far


@pytest.mark.parametrize("h", [0xFFFE, 0xFFFF, 0x10000, 70000])
def test_window_limit_chains(h):
    img = window_chain(h)
    g, e = orc.GBWT.load(img.array), HostSim(img.array)
    longest, far = window_limits(e)
    assert longest == h    # anchor records of exactly h positions, on both sides of the staging limit
    if h == 70000:
        assert far > 0     # allele records whose offset into the next anchor does not fit 16 bits
    for k in (2, 17, 32):
        pats = synth.patterns(CHAIN_SITES, h, CHAIN_SEED, n=3000, k=k, **CHAIN_MODEL)
        assert pc.states_equal(e.find_extend(pats), g.find_extend_batch(pats))
    ids = np.arange(0, 2 * h, 997, dtype=np.uint64)
    assert np.array_equal(e.sequence_lengths(ids), g.sequence_lengths(ids))
    o_off, o_nodes = g.extract_batch(ids)
    offsets, nodes, _ = e.extract(ids)
    assert np.array_equal(offsets, o_off) and np.array_equal(nodes, o_nodes)


# The rows of the extraction window hold node - row_base in 16 signed bits (find_window.cu: fits_row accepts
# [-0x8000, 0x7FFF]). Inside one window two nodes never differ by that much; a row spans a larger difference only when a
# lane starts a round below the window, takes its one step from the global layout and lands inside the window. A window
# sits above a lane only when more lanes walk towards lower records than towards higher ones: it is then placed from the
# highest lane.
ROW_JUMPS = (0x7FFF, 0x8000, 0x8001, 0xFFFF, 0x10000, 0x17FFF, 0x18000)
ROW_TOP = 0x40000        # id of the node every walk down starts from


def row_jump_paths(copies=12, length=24):
    """`copies` paths that walk down through reverse-orientation nodes at ids ROW_TOP, ROW_TOP - 1, ... and then up
    through forward nodes at low ids, so that both strands of each start walking down; and for every jump d one path
    that starts on the node d below the top node and steps up to it."""
    down = [2 * (ROW_TOP - t) + 1 for t in range(length)]
    up = [2 * (0x1000 + t) for t in range(length)]
    return [down + up for _ in range(copies)] + [[down[0] - d] + down for d in ROW_JUMPS]


def row_jump_starts(paths):
    """(first node of every sequence, walking down?) of the bidirectional index of `paths`."""
    firsts = [s[0] for s in gb.bidirectional_sequences(paths)]
    return firsts, [x & 1 == 1 for x in firsts]


def test_row_jumps():
    paths = row_jump_paths()
    firsts, down = row_jump_starts(paths)
    assert 2 * sum(down) > len(down)   # the first window is placed from the highest lane
    top = 2 * ROW_TOP + 1
    assert max(firsts) == top and [top - p[0] for p in paths if p[0] != top] == list(ROW_JUMPS)
    assert all(p[1] == top for p in paths if p[0] != top)
    img, _ = bwt_image(paths)
    g, e = orc.GBWT.load(img), HostSim(img)
    check_graph_index(e, g, paths)


# ---- D. node-id distances and large ids ------------------------------------------------------------------------------

ID_JUMPS = [1, 0x3FFF, 0x4000, 0x4001, 0x8000, -0x4000, -0x4001, 2, -0x3FFF, 5]


def far_jump_paths(haplotypes=48, length=60, seed=5, detour=0.3):
    """Paths over a chain whose consecutive node ids jump by about +-0x4000, 0x8000 and once by 2^20, with a third of
    the nodes in reverse orientation: GBWT node differences around +-0x8000 (the signed 16-bit rows of the extraction
    windows), 0x10000 and 2^21. Each chain position has a detour node, taken with probability `detour`."""
    rng = random.Random(seed)
    base = 0x30000
    used, main, alt = set(), [], []
    cur = base
    for j in range(length):
        cur += (1 << 20) if j == length // 2 else ID_JUMPS[j % len(ID_JUMPS)]
        while cur in used or cur + 7 in used or cur <= base:
            cur += 3
        used.update((cur, cur + 7))
        o = 1 if j % 3 == 2 else 0
        main.append(2 * cur + o); alt.append(2 * (cur + 7) + o)
    paths = [[2 * base]]   # (the smallest id, forward: the alphabet offset stays odd)
    for _ in range(haplotypes):
        paths.append([alt[j] if rng.random() < detour else main[j] for j in range(length)])
    return paths


def node_steps(paths):
    return {b - a for p in paths for a, b in zip(p, p[1:])}


def bwt_image(paths, shift=0, extra_records=0):
    seqs = gb.bidirectional_sequences([[x + shift for x in p] for p in paths])
    b = gb.build_bwt(seqs)
    starts, data = list(b["starts"]), b["data"] + b"\x00" * extra_records
    starts += [len(b["data"]) + i for i in range(extra_records)]
    img = synth.gbwt_image(b["sequences"], b["size"], b["offset"], b["alphabet_size"] + extra_records, 5, starts, data)
    return img, b


@pytest.fixture(scope="module")
def far_jump_index():
    paths = far_jump_paths()
    img, b = bwt_image(paths)
    return paths, img, b


def check_graph_index(e, g, paths, sample=0):
    ids = np.arange(g.sequences() + 2, dtype=np.uint64)
    assert np.array_equal(e.sequence_lengths(ids), g.sequence_lengths(ids))
    o_off, o_nodes = g.extract_batch(ids)
    offsets, nodes, _ = e.extract(ids)
    assert np.array_equal(offsets, o_off) and np.array_equal(nodes, o_nodes)
    seqs = [p for p in pc.all_sequences(g) if p]
    for k in (1, 2, 5, 17):
        pats = np.array(pc.subpath_patterns(seqs, k), dtype=np.uint64)
        want = g.find_extend_batch(pats)
        assert np.all(want["end"] > want["start"])
        assert pc.states_equal(e.find_extend(pats), want)
    args = pc.bd_triples([s[:6] for s in seqs[:: max(1, len(seqs) // 12)]])
    assert pc.states_equal(e.bd_search(*args), g.bd_search_batch(*args))


def test_far_node_jumps(far_jump_index):
    paths, img, b = far_jump_index
    steps = node_steps(paths)
    assert {0x8000, 0x8002}.issubset(steps) and any(s > 2**21 for s in steps)
    assert any(-0x8002 <= s <= -0x8000 for s in steps) and any(0x7FFE <= s <= 0x7FFF for s in steps)
    g, e = orc.GBWT.load(img), HostSim(img)
    assert e.records() > 2**21
    check_graph_index(e, g, paths)


def large_id_shift(paths):
    """Even shift that puts the largest node (a reverse orientation) at 2^32 - 3; one empty record more makes the
    alphabet 2^32 - 1."""
    top = max(x | 1 for p in paths for x in p)
    return 2**32 - 3 - top


def test_large_node_ids(far_jump_index):
    paths, _, _ = far_jump_index
    shift = large_id_shift(paths)
    img, b = bwt_image(paths, shift, extra_records=1)
    assert b["alphabet_size"] + 1 == U32MAX and b["offset"] >= 2**32 - 2**22 and b["offset"] & (1 << 31)
    g, e = orc.GBWT.load(img), HostSim(img)
    check_graph_index(e, g, paths)
    # u64 patterns with a real node plus 2^32 at one position: None, never the node it would alias in 32 bits
    seqs = [p for p in pc.all_sequences(g) if len(p) >= 4]
    pats = np.array([s[:4] for s in seqs], dtype=np.uint64)
    for col in range(4):
        bad = pats.copy()
        bad[:, col] += np.uint64(2**32)
        assert pc.states_equal(e.find_extend(bad), g.find_extend_batch(bad))
        assert not np.any(g.find_extend_batch(bad)["end"])
    # two records more: node 2^32 - 1 is in the alphabet (its id still fits 32 bits); three: the alphabet passes 2^32
    img2, _ = bwt_image(paths, shift, extra_records=2)
    g2, e2 = orc.GBWT.load(img2), HostSim(img2)
    assert g2.alphabet_size() == 2**32 and e2.records() == 2**32 - g2.alphabet_offset()
    nodes = np.array([0, g2.alphabet_offset(), g2.alphabet_offset() + 1, 2**32 - 3, 2**32 - 2, 2**32 - 1, 2**32, 2**32 + 1],
                     dtype=np.uint64)
    assert pc.states_equal(e2.find(nodes), g2.find_batch(nodes))
    assert pc.states_equal(e2.find_extend(pats), g2.find_extend_batch(pats))
    img3, _ = bwt_image(paths, shift, extra_records=3)
    assert orc.GBWT.load(img3).alphabet_size() == 2**32 + 1
    with pytest.raises(IOError, match="32-bit"):
        HostSim(img3)
