"""The device-pointer entry points (gbwt_b200_*_device) through the C ABI, bit for bit against the oracle and against
their host twins on the same input: every search schedule on dense and run-length bubble chains, ragged and
bidirectional batches called on a slice of a larger device batch (d_offsets[0] > 0), extension in place, follow with
counts only and with truncated slots that start above 0, extraction into slots that start above 0, the caller's side
stream and stream 0, and the contracts of a unidirectional index and of empty batches."""
import os
import re

import numpy as np
import pytest

import gbwt_builder as gb
import parity_checks as pc
from oracle import oracle as orc
from synth import synth
from test_gpu_window import damaged_batches, image_of

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
U64MAX = np.uint64(2**64 - 1)
SENTINEL = 0xAB
THREADS = orc.max_threads()

MODELS = {"dense": dict(), "tri-allelic": dict(alt_ppm=50_000, tri_mod=4)}
# GBWT_B200_* knobs of each search schedule: the plain kernels (lean, general, general with runs, lean mixed), the
# locality sort without windows, and the record windows with one-pass placement or the exact sort
SCHEDULES = {
    "lean": dict(LOCALITY=0),
    "general": dict(LOCALITY=0, FIND_LEAN=0),
    "general-runs": dict(LOCALITY=0, FIND_LEAN=2),
    "lean-mixed": dict(LOCALITY=0, FIND_LEAN=3),
    "sorted": dict(LOCALITY=1, FIND_WINDOW=0),
    "windows-direct": dict(LOCALITY=1, FIND_WINDOW=2, WINDOW_STATS=1, WINDOW_DIRECT=1),
    "windows-sorted": dict(LOCALITY=1, FIND_WINDOW=2, WINDOW_STATS=1, WINDOW_DIRECT=0),
}
S, H, SEED = 1500, 64, 7


@pytest.fixture(scope="module")
def b200():
    import gbwt_rs_b200
    return gbwt_rs_b200


@pytest.fixture(scope="module")
def chains(b200):
    out = {}
    for name, model in MODELS.items():
        img = synth.bubble_chain(S, H, SEED, **model)
        out[name] = (orc.GBWT.load(img.array), b200.GBWT.from_bytes(img.array), model)
    return out


# ---- device buffers and streams ---------------------------------------------------------------------------------------

def dev(a):
    """A device copy of a numpy array (as bytes)."""
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8).copy()).cuda()


def filled(n_bytes):
    import torch
    return torch.full((max(n_bytes, 1),), SENTINEL, dtype=torch.uint8, device="cuda")


def host(t, dtype, count=None):
    a = t.cpu().numpy().view(dtype)
    return a if count is None else a[:count]


def ptr(t, skip_bytes=0):
    return None if t is None else t.data_ptr() + skip_bytes


def streams():
    """A side stream of the caller's and stream 0."""
    import torch
    return [torch.cuda.Stream(), None]


def run_on(b200, stream, call):
    """Enqueues call(stream handle) on `stream` once the inputs are in place, and waits for that stream only."""
    import torch
    torch.cuda.synchronize()
    rc = call(stream.cuda_stream if stream is not None else 0)
    assert rc == 0, b200.library().gbwt_b200_last_error().decode()
    (stream if stream is not None else torch.cuda.default_stream()).synchronize()


def ragged_batch(pats, rng, prefix=5):
    """Patterns of 0 to k nodes cut from `pats` (runs of empty ones included), in one node array that starts with
    `prefix` nodes no pattern uses: offsets[0] == prefix."""
    n, k = pats.shape
    lens = rng.choice([0, 1, 2, 9, k // 2, k], size=n)
    lens[n // 4:n // 4 + 9] = 0
    lens[-3:] = 0
    nodes = [np.full(prefix, 2**40, dtype=np.uint64)] + [pats[q, :lens[q]] for q in range(n)]
    offsets = np.zeros(n + 1, dtype=np.uint64)
    offsets[0] = prefix
    offsets[1:] = prefix + np.cumsum(lens)
    return np.concatenate(nodes), offsets


def bd_triples(offsets, rng):
    lens = np.diff(offsets)
    n = len(lens)
    first = (lens * rng.random(n)).astype(np.uint64)
    start = (first * rng.random(n)).astype(np.uint64)
    end = np.minimum(lens, first + 1 + ((lens - first) * rng.random(n)).astype(np.uint64)).astype(np.uint64)
    first[lens == 0] = start[lens == 0] = end[lens == 0] = 0
    return first, start, end


def bd_search_oracle(g, nodes, offsets, first, start, end):
    """The oracle's answers where the header admits the search (start <= first < end <= len); None elsewhere, which is what
    the library answers there (the oracle would read the path at `first` regardless)."""
    valid = (start <= first) & (first < end) & (end <= np.diff(offsets))
    want = np.zeros(len(first), orc.BDSTATE_DTYPE)
    at = np.append(offsets[:-1][valid], offsets[-1])   # (the oracle reads path q from nodes + offsets[q])
    want[valid] = g.bd_search_batch(nodes, at, first[valid], start[valid], end[valid], threads=THREADS)
    return want


# ---- search schedules -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("schedule", list(SCHEDULES))
@pytest.mark.parametrize("model", list(MODELS))
def test_search_device_calls(b200, chains, model, schedule, monkeypatch):
    """find_extend(_u32)_device for pattern lengths 0 .. 33, and find_extend_ragged_device / bd_search_device on a batch
    and on its slice from row q0 (d_offsets + q0): the oracle, the host twin and the rows q0.. of the full call agree."""
    for k, v in SCHEDULES[schedule].items():
        monkeypatch.setenv("GBWT_B200_" + k, str(v))
    g, e, params = chains[model]
    lib = b200.library()
    rng = np.random.default_rng(11)
    queries_before = e.window_info()["queries"]
    for k in (0, 1, 2, 31, 32, 33):
        if k == 0:
            pats = np.zeros((700, 0), dtype=np.uint64)
            want = np.zeros(len(pats), orc.STATE_DTYPE)
        else:
            pats = np.concatenate(damaged_batches(g, synth.patterns(S, H, SEED, n=3000, k=k, **params), rng))
            want = g.find_extend_batch(pats, threads=THREADS)
        narrow = np.all(pats < 2**32, axis=1)
        p32 = pats[narrow].astype(np.uint32)
        assert pc.states_equal(e.find_extend(pats), want) and pc.states_equal(e.find_extend_u32(p32), want[narrow])
        for stream in streams():
            d_p, d_p32 = (dev(pats), dev(p32)) if k else (filled(16), filled(16))   # (k == 0 reads no pattern)
            d_out, d_out32 = filled(24 * len(pats)), filled(24 * len(p32))
            run_on(b200, stream, lambda s: lib.gbwt_b200_find_extend_device(e._h, ptr(d_p), len(pats), k, ptr(d_out), s))
            run_on(b200, stream, lambda s: lib.gbwt_b200_find_extend_u32_device(e._h, ptr(d_p32), len(p32), k, ptr(d_out32), s))
            assert pc.states_equal(host(d_out, orc.STATE_DTYPE), want), k
            assert pc.states_equal(host(d_out32, orc.STATE_DTYPE), want[narrow]), k
    # ragged and bidirectional batches, whole and sliced
    pats = np.concatenate(damaged_batches(g, synth.patterns(S, H, SEED, n=5000, k=40, seed_q=3, **params), rng))
    nodes, offsets = ragged_batch(pats, rng)
    first, start, end = bd_triples(offsets, rng)
    n, q0 = len(offsets) - 1, len(offsets) // 3
    want = g.find_extend_ragged(nodes, offsets, threads=THREADS)
    bd_want = bd_search_oracle(g, nodes, offsets, first, start, end)
    assert np.count_nonzero(want["end"] > want["start"]) > n // 4
    assert np.count_nonzero(bd_want["forward"]["end"] > bd_want["forward"]["start"]) > n // 4
    assert pc.states_equal(e.find_extend_ragged(nodes, offsets), want)
    assert pc.states_equal(e.bd_search(nodes, offsets, first, start, end), bd_want)
    d_nodes, d_offsets, d_first, d_start, d_end = map(dev, (nodes, offsets, first, start, end))
    for stream in streams():
        for row in (0, q0):
            d_out, d_bd = filled(24 * (n - row)), filled(48 * (n - row))
            run_on(b200, stream, lambda s: lib.gbwt_b200_find_extend_ragged_device(e._h, ptr(d_nodes), ptr(d_offsets, 8 * row), n - row, ptr(d_out), s))
            run_on(b200, stream, lambda s: lib.gbwt_b200_bd_search_device(e._h, ptr(d_nodes), ptr(d_offsets, 8 * row), ptr(d_first, 8 * row),
                                                                           ptr(d_start, 8 * row), ptr(d_end, 8 * row), n - row, ptr(d_bd), s))
            assert pc.states_equal(host(d_out, orc.STATE_DTYPE), want[row:]), row
            assert pc.states_equal(host(d_bd, orc.BDSTATE_DTYPE), bd_want[row:]), row
    if "windows" in schedule:
        assert e.window_info()["queries"] > queries_before   # the batches went through the record windows


# ---- single steps, in place, follow, extraction -----------------------------------------------------------------------

def search_inputs(g, params, rng, n):
    """Nodes to find (every id, random ones, far ones), and (head, next) pairs: half of them consecutive nodes of a path,
    half random."""
    lo, hi = max(0, g.alphabet_offset() - 2), g.alphabet_size() + 3
    nodes = np.concatenate([np.arange(g.alphabet_size() + 2, dtype=np.uint64), rng.integers(lo, hi, n, dtype=np.uint64),
                            np.array([2**32 - 1, 2**32, 2**63, 2**64 - 1], dtype=np.uint64)])
    m = len(nodes)
    pairs = synth.patterns(S, H, SEED, n=m // 2, k=2, seed_q=13, **params)
    heads = np.concatenate([pairs[:, 0], rng.integers(g.first_node(), g.alphabet_size(), m - m // 2, dtype=np.uint64)])
    tails = np.concatenate([pairs[:, 1], rng.integers(lo, hi, m - m // 2, dtype=np.uint64)])
    return nodes, heads, tails


@pytest.mark.parametrize("model", list(MODELS))
def test_step_device_calls(b200, chains, model):
    """find / extend / bd_find / bd_extend (both directions) / forward: device call = oracle = host twin; extend_device and
    bd_extend_device with d_out == d_states."""
    g, e, params = chains[model]
    lib = b200.library()
    rng = np.random.default_rng(5)
    nodes, heads, nxt = search_inputs(g, params, rng, 30_000)
    n = len(nodes)
    states = g.find_batch(heads, threads=THREADS)
    want_find, want_ext = g.find_batch(nodes, threads=THREADS), g.extend_batch(states, nxt, threads=THREADS)
    bd = g.bd_find_batch(nodes, threads=THREADS)
    bd_states = g.bd_find_batch(heads, threads=THREADS)
    want_bd = [g.bd_extend_batch(bd_states, nxt, backward=b, threads=THREADS) for b in (False, True)]
    positions = np.zeros(n, orc.POS_DTYPE)
    positions["node"] = nodes
    positions["offset"] = rng.integers(0, 2 * H + 2, n)
    want_fwd = g.forward_batch(positions, threads=THREADS)
    assert pc.states_equal(e.find(nodes), want_find) and pc.states_equal(e.extend(states, nxt), want_ext)
    assert pc.states_equal(e.bd_find(nodes), bd) and pc.states_equal(e.forward(positions), want_fwd)
    assert pc.states_equal(e.extend_forward(bd_states, nxt), want_bd[0]) and pc.states_equal(e.extend_backward(bd_states, nxt), want_bd[1])
    assert np.count_nonzero(want_ext["end"] > want_ext["start"]) > n // 4
    d_nodes, d_nxt, d_pos = dev(nodes), dev(nxt), dev(positions)
    for stream in streams():
        d_out, d_bd, d_fwd = filled(24 * n), filled(48 * n), filled(16 * n)
        run_on(b200, stream, lambda s: lib.gbwt_b200_find_device(e._h, ptr(d_nodes), n, ptr(d_out), s))
        run_on(b200, stream, lambda s: lib.gbwt_b200_bd_find_device(e._h, ptr(d_nodes), n, ptr(d_bd), s))
        run_on(b200, stream, lambda s: lib.gbwt_b200_forward_device(e._h, ptr(d_pos), n, ptr(d_fwd), s))
        assert pc.states_equal(host(d_out, orc.STATE_DTYPE), want_find)
        assert pc.states_equal(host(d_bd, orc.BDSTATE_DTYPE), bd)
        assert pc.states_equal(host(d_fwd, orc.POS_DTYPE), want_fwd)
        d_st = dev(states)   # in place
        run_on(b200, stream, lambda s: lib.gbwt_b200_extend_device(e._h, ptr(d_st), ptr(d_nxt), n, ptr(d_st), s))
        assert pc.states_equal(host(d_st, orc.STATE_DTYPE), want_ext)
        for backward in (0, 1):
            d_bst = dev(bd_states)
            run_on(b200, stream, lambda s: lib.gbwt_b200_bd_extend_device(e._h, ptr(d_bst), ptr(d_nxt), n, backward, ptr(d_bst), s))
            assert pc.states_equal(host(d_bst, orc.BDSTATE_DTYPE), want_bd[backward])


def slot_offsets(sizes, first, pattern=(1.0, 0.5, 0.0, 2.0)):
    """Output slots that start at `first`: exact, half, empty and over-long (+3) in turn, and a run of empty ones."""
    n = len(sizes)
    caps = np.array([int(int(s) * pattern[i % 4]) + (3 if pattern[i % 4] > 1 else 0) for i, s in enumerate(sizes)], dtype=np.uint64)
    caps[n // 3:n // 3 + 8] = 0
    offsets = np.zeros(n + 1, dtype=np.uint64)
    offsets[0] = first
    offsets[1:] = first + np.cumsum(caps)
    return offsets


def check_slots(out_bytes, dtype, offsets, truth, item_of=None):
    """Result i (truth(i), an array of `dtype`) cut to slot i; the bytes before the first slot and after the last one hold
    the sentinel."""
    w = np.dtype(dtype).itemsize
    lo, hi = int(offsets[0]), int(offsets[-1])
    assert np.all(out_bytes[:lo * w] == SENTINEL) and np.all(out_bytes[hi * w:] == SENTINEL)
    out = out_bytes[:hi * w].view(dtype)
    for i in range(len(offsets) - 1):
        a, b = int(offsets[i]), int(offsets[i + 1])
        t = truth(i)
        m = min(b - a, len(t))
        assert out[a:a + m].tobytes() == t[:m].tobytes(), i


@pytest.mark.parametrize("backward", [0, 1])
def test_follow_device(b200, chains, backward):
    """follow_device: counts only (d_out = NULL), then into slots that start above 0 and are exact, truncated, empty or
    over-long, on a slice of the state batch: counts in full, each slot holds the first extensions, and nothing before,
    after or behind the written extensions changes."""
    g, e, _ = chains["tri-allelic"]
    lib = b200.library()
    rng = np.random.default_rng(9 + backward)
    states = g.bd_find_batch(np.arange(g.alphabet_size() + 3, dtype=np.uint64), threads=THREADS)
    states = np.concatenate([states, g.bd_extend_batch(states[rng.integers(0, len(states), 3000)], rng.integers(0, g.alphabet_size(), 3000, dtype=np.uint64),
                                                       backward=bool(backward), threads=THREADS)])
    w_off, want, counts = g.follow_batch(states, backward=bool(backward), threads=THREADS)
    assert np.any(counts > 1)
    h_off, h_out, h_counts = e.follow(states, bool(backward))
    assert np.array_equal(h_counts, counts) and pc.states_equal(h_out, want)
    sizes = np.where(counts == U64MAX, np.uint64(0), counts)
    q0 = 100
    slots = slot_offsets(sizes[q0:], first=40)
    n = len(states)
    d_states = dev(states)
    d_slots = dev(np.concatenate([np.zeros(q0, np.uint64), slots]))   # the call gets d_slots + q0
    for stream in streams():
        d_counts = filled(8 * n)
        run_on(b200, stream, lambda s: lib.gbwt_b200_follow_device(e._h, ptr(d_states), n, backward, None, None, ptr(d_counts), s))
        assert np.array_equal(host(d_counts, np.uint64), counts)
        d_out, d_counts = filled(48 * (int(slots[-1]) + 20)), filled(8 * (n - q0))
        run_on(b200, stream, lambda s: lib.gbwt_b200_follow_device(e._h, ptr(d_states, 48 * q0), n - q0, backward, ptr(d_slots, 8 * q0),
                                                                     ptr(d_out), ptr(d_counts), s))
        assert np.array_equal(host(d_counts, np.uint64), counts[q0:])
        got = d_out.cpu().numpy()
        check_slots(got, orc.BDSTATE_DTYPE, slots, lambda i: want[int(w_off[q0 + i]):int(w_off[q0 + i + 1])])
        for i in range(n - q0):   # the device call writes only the extensions it has
            a = int(slots[i]) + min(int(sizes[q0 + i]), int(slots[i + 1] - slots[i]))
            assert np.all(got[48 * a:48 * int(slots[i + 1])] == SENTINEL), i


def test_extract_device_into_slots_above_zero(b200, chains):
    """extract_device with d_out_offsets[0] > 0 and slots of every kind, on checkpointed and plain indexes and for
    sequences whose lengths are known (two-ended walks): the oracle's paths at the right slots, lengths in full."""
    g, _, params = chains["dense"]
    lib = b200.library()
    img = synth.bubble_chain(S, H, SEED, **params)
    ids = np.concatenate([np.arange(2 * H, dtype=np.uint64), np.array([2 * H, 2**40], dtype=np.uint64)])
    o_off, o_nodes = g.extract_batch(ids, threads=THREADS)
    lengths = g.sequence_lengths(ids, threads=THREADS)
    slots = slot_offsets(np.diff(o_off), first=1000)
    d_ids, d_slots = dev(ids), dev(slots)
    for ckpt in (True, False):
        e = b200.GBWT.from_bytes(img.array, checkpoints=ckpt)
        for measured in (False, True):
            if measured:
                assert np.array_equal(e.sequence_lengths(ids), lengths)
            for stream in streams():
                d_out, d_len = filled(8 * (int(slots[-1]) + 50)), filled(8 * len(ids))
                run_on(b200, stream, lambda s: lib.gbwt_b200_extract_device(e._h, ptr(d_ids), len(ids), ptr(d_slots), ptr(d_out), ptr(d_len), s))
                assert np.array_equal(host(d_len, np.uint64), lengths)
                check_slots(d_out.cpu().numpy(), np.uint64, slots, lambda i: o_nodes[int(o_off[i]):int(o_off[i + 1])])


# ---- contracts ----------------------------------------------------------------------------------------------------------

def test_unidirectional_index_launches_nothing(b200):
    """The bidirectional device calls and follow_device on a unidirectional index: GBWT_B200_E_NOT_BIDIRECTIONAL, no
    kernel, the output untouched."""
    import torch
    paths = [[2, 4, 6], [2, 6], [4, 6, 2, 4]]
    img = image_of(gb.build_bwt(gb.bidirectional_sequences(paths)), bidirectional=False)
    e = b200.GBWT.from_bytes(img)
    assert not e.is_bidirectional()
    lib = b200.library()
    n = 4
    d_nodes, d_offsets, d_idx = dev(np.array([2, 4, 6, 2], np.uint64)), dev(np.arange(n + 1, dtype=np.uint64)), dev(np.zeros(n, np.uint64))
    d_states = dev(np.zeros(n, orc.BDSTATE_DTYPE))
    calls = {
        "bd_find": lambda out, s: lib.gbwt_b200_bd_find_device(e._h, ptr(d_nodes), n, ptr(out), s),
        "bd_extend": lambda out, s: lib.gbwt_b200_bd_extend_device(e._h, ptr(d_states), ptr(d_nodes), n, 0, ptr(out), s),
        "bd_search": lambda out, s: lib.gbwt_b200_bd_search_device(e._h, ptr(d_nodes), ptr(d_offsets), ptr(d_idx), ptr(d_idx), ptr(d_idx), n, ptr(out), s),
        "follow": lambda out, s: lib.gbwt_b200_follow_device(e._h, ptr(d_states), n, 0, ptr(d_offsets), ptr(out), ptr(d_idx), s),
    }
    for name, call in calls.items():
        for stream in streams():
            out = filled(48 * n)
            torch.cuda.synchronize()
            before = b200.kernel_launches()
            assert call(out, stream.cuda_stream if stream is not None else 0) == b200.E_NOT_BIDIRECTIONAL, name
            torch.cuda.synchronize()
            assert b200.kernel_launches() == before, name
            assert np.all(out.cpu().numpy() == SENTINEL), name
    assert np.all(host(d_idx, np.uint64) == 0)


EMPTY_CALLS = {   # every device entry point with an empty batch and NULL pointers
    "find_extend_device": lambda h: (h, None, 0, 32, None),
    "find_extend_u32_device": lambda h: (h, None, 0, 32, None),
    "find_extend_ragged_device": lambda h: (h, None, None, 0, None),
    "find_device": lambda h: (h, None, 0, None),
    "extend_device": lambda h: (h, None, None, 0, None),
    "bd_find_device": lambda h: (h, None, 0, None),
    "bd_extend_device": lambda h: (h, None, None, 0, 1, None),
    "bd_search_device": lambda h: (h, None, None, None, None, None, 0, None),
    "follow_device": lambda h: (h, None, 0, 0, None, None, None),
    "forward_device": lambda h: (h, None, 0, None),
    "sequence_lengths_device": lambda h: (h, None, 0, None),
    "extract_device": lambda h: (h, None, 0, None, None, None),
    "locate_device": lambda h: (h, None, 0, None),
    "locate_states_device": lambda h: (h, None, 0, None, None, None),
    "dna_lengths_device": lambda h: (h, None, 0, None),
    "extract_dna_device": lambda h: (h, None, 0, 0, None, None, None),
}


def test_empty_batches_launch_nothing(b200):
    """n == 0 with NULL pointers: GBWT_B200_OK and no kernel, for every device entry point the header declares (on an
    index that has a graph and locate samples, so that no check on the index stops the call first)."""
    import torch
    declared = set(re.findall(r"\bgbwt_b200_(\w+_device)\(", open(os.path.join(ROOT, "include", "gbwt_b200.h")).read()))
    assert declared == set(EMPTY_CALLS)
    e = b200.GBWT.load(os.path.join(GOLDEN, "example.gbz"), locate=True)
    assert e.has_graph() and e.locate_info()["present"] and e.is_bidirectional()
    lib = b200.library()
    side = torch.cuda.Stream()
    for name, args in EMPTY_CALLS.items():
        for stream in (side.cuda_stream, 0):
            before = b200.kernel_launches()
            assert getattr(lib, "gbwt_b200_" + name)(*args(e._h), stream) == 0, (name, lib.gbwt_b200_last_error().decode())
            assert b200.kernel_launches() == before, name
    torch.cuda.synchronize()
