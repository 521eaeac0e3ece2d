"""Building a GBWT from paths on the GPU (gbwt_b200_build_image, include/gbwt_b200_build.h) against the definition in
tests/gbwt_builder.py, the reference's fixtures and the closed-form bubble chains of synth/.

The image must be byte for byte what from_parts(<the builder's header and records>).serialize() writes. The long-path case
is too long for the brute-force builder (its keys are whole reversed prefixes), so there the built index is checked through
the oracle: every sequence comes back, and every sampled subpath has its brute-force count."""
import os
import random

import numpy as np
import pytest

import gbwt_builder as gbb
import golden_vectors as gv
from oracle import oracle as orc
from synth import synth

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
U32 = 1 << 32


@pytest.fixture(scope="module")
def b200():
    import gbwt_rs_b200
    return gbwt_rs_b200


def expected_image(b200, paths, bidirectional=True):
    b = gbb.build_bwt(gbb.bidirectional_sequences(paths) if bidirectional else [list(p) for p in paths])
    ix = b200.GBWT.from_parts(b["sequences"], b["size"], b["offset"], b["alphabet_size"], 1 if bidirectional else 0,
                              b["data"], b["starts"])
    return ix.serialize(), b


def same_bwt(image, data, starts, fields):
    g = orc.GBWT.load(image)
    assert g.bwt_data() == data
    assert [int(x) for x in g.record_starts()] == [int(x) for x in starts]
    assert (g.alphabet_offset(), g.alphabet_size(), g.sequences(), g.len()) == fields


@pytest.mark.parametrize("name,paths", [
    ("example.gbwt", gv.true_paths(False)),
    ("with-empty.gbwt", gv.true_paths(True)),
    ("translation.gbwt", gv.TRANSLATION_PATHS),
])
def test_fixtures(b200, name, paths):
    image = b200.build_image(paths, bidirectional=True)
    g = orc.GBWT.load(os.path.join(GOLDEN, name))
    same_bwt(image, g.bwt_data(), g.record_starts(), (g.alphabet_offset(), g.alphabet_size(), g.sequences(), g.len()))
    assert orc.GBWT.load(image).is_bidirectional()
    want, _ = expected_image(b200, paths)
    assert image == want


def test_only_empty_paths(b200):
    for bidirectional in (True, False):
        image = b200.build_image([[], [], []], bidirectional=bidirectional)
        want, b = expected_image(b200, [[], [], []], bidirectional)
        assert image == want and len(b["starts"]) == 1


def random_paths(rng, kind):
    """Small path sets for the brute-force builder. Nodes are >= 2 so that both orientations are valid."""
    n_nodes = rng.choice([2, 3, 6, 12, 40])
    walk = lambda length: [2 * rng.randint(1, n_nodes) + (1 if rng.random() < 0.3 else 0) for _ in range(length)]
    paths = [walk(rng.randint(0, rng.choice([3, 8, 20]))) for _ in range(rng.choice([1, 3, 10, 40]))]
    if kind == "duplicates":
        paths += [list(p) for p in rng.sample(paths, max(1, len(paths) // 2))] * 2
    elif kind == "prefixes":
        paths += [p[:rng.randint(0, len(p))] for p in paths]
    elif kind == "short":
        paths += [[], [2 * rng.randint(1, n_nodes)], [], [2 * rng.randint(1, n_nodes) + 1]]
    elif kind == "wide":  # sigma >= 255 in record 0 and in the shared first node
        paths += [[4, 2 * k] for k in range(3, 3 + rng.choice([254, 255, 300]))]
    elif kind == "long_runs":  # runs above 256 / sigma
        paths += [[6, 8, 10]] * rng.choice([100, 300]) + [[6, 9, 10]] * 40
    elif kind == "sparse":  # many empty records
        paths = [[x * 1000 + (x & 1) for x in p] for p in paths]
    elif kind == "high":  # ids packed just below 2^32
        paths = [[U32 - 2 * n_nodes - 4 + x for x in p] for p in paths]
    rng.shuffle(paths)
    if not any(paths):
        paths.append([2, 4, 2])
    return paths


KINDS = ["plain", "duplicates", "prefixes", "short", "wide", "long_runs", "sparse", "high"]


@pytest.mark.parametrize("bidirectional", [True, False])
@pytest.mark.parametrize("kind", KINDS)
def test_random_paths_against_builder(b200, kind, bidirectional):
    rng = random.Random(f"{kind}-{bidirectional}")
    for _ in range(6):
        paths = random_paths(rng, kind)
        info = {}
        image = b200.build_image(paths, bidirectional=bidirectional, info=info)
        want, b = expected_image(b200, paths, bidirectional)
        assert image == want
        assert info["positions"] == b["size"] and info["peak_device_bytes"] > 0


def test_unidirectional_accepts_node_1(b200):
    paths = [[1, 2, 1, 3], [3, 1], []]
    image = b200.build_image(paths, bidirectional=False)
    assert image == expected_image(b200, paths, False)[0]


def brute_count(seqs, pattern):
    k, total = len(pattern), 0
    for s in seqs:
        if len(s) >= k:
            w = np.lib.stride_tricks.sliding_window_view(s, k)
            total += int(np.all(w == pattern, axis=1).sum())
    return total


@pytest.mark.parametrize("bidirectional", [True, False])
def test_one_long_path(b200, bidirectional):
    """About 10^5 nodes of a repeated cycle with a few detours: contexts stay equal for long stretches, so the doubling takes
    many rounds."""
    rng = np.random.default_rng(5)
    cycle = np.array([2, 4, 6, 8, 10, 12, 14], dtype=np.uint64)
    path = np.tile(cycle, 100_000 // len(cycle))
    path[rng.choice(len(path), 20, replace=False)] = 16
    paths = [path, path[:5000].copy()]
    info = {}
    image = b200.build_image(paths, bidirectional=bidirectional, info=info)
    assert info["rounds"] >= 10
    g = orc.GBWT.load(image)
    seqs = [np.asarray(p, dtype=np.uint64) for p in (gbb.bidirectional_sequences([list(map(int, p)) for p in paths])
                                                     if bidirectional else paths)]
    assert g.sequences() == len(seqs) and g.len() == sum(len(s) + 1 for s in seqs)
    for i, s in enumerate(seqs):
        assert np.array_equal(np.asarray(g.sequence(i), dtype=np.uint64), s)
    pats = []
    for _ in range(200):
        s = seqs[int(rng.integers(len(seqs)))]
        k = int(rng.integers(1, 40))
        j = int(rng.integers(0, len(s) - k))
        pats.append(s[j:j + k])
    for p in pats:
        st = g.find(int(p[0]))
        for x in p[1:]:
            st = g.extend(st, int(x)) if st is not None else None
        assert (0 if st is None else st[2] - st[1]) == brute_count(seqs, p)
    assert b200.build_image(paths, bidirectional=bidirectional) == image


def chain_paths(S, H, seed, **kw):
    return [synth.sequence(S, H, seed, 2 * h, **kw) for h in range(H)]


@pytest.mark.parametrize("S,H,seed,kw", [
    (1, 1, 0, {}), (7, 9, 3, {}), (500, 64, 42, {}), (2000, 33, 4, {}),
    (500, 64, 42, dict(alt_ppm=50_000, tri_mod=5)), (3000, 100, 9, dict(alt_ppm=200_000, tri_mod=3)),
])
def test_bubble_chains(b200, S, H, seed, kw):
    img = synth.bubble_chain(S, H, seed, **kw)
    g = orc.GBWT.load(img.array)
    image = b200.build_image(chain_paths(S, H, seed, **kw), bidirectional=True)
    same_bwt(image, g.bwt_data(), g.record_starts(), (g.alphabet_offset(), g.alphabet_size(), g.sequences(), g.len()))


def test_large_bubble_chain_from_device_paths(b200):
    """333 333 sites x 256 haplotypes (341 M positions, well beyond L2): the paths are extracted on the device from the synth
    image and built from there with no host round trip."""
    import torch
    S, H, seed = 333_333, 256, 42
    img = synth.bubble_chain(S, H, seed)
    ix = b200.GBWT.from_bytes(img.array)
    L = 2 * S + 1
    ids = torch.arange(0, 2 * H, 2, dtype=torch.int64, device="cuda")
    offsets = torch.arange(0, H + 1, dtype=torch.int64, device="cuda") * L
    nodes = torch.empty(H * L, dtype=torch.int64, device="cuda")
    lengths = torch.empty(H, dtype=torch.int64, device="cuda")
    ix.extract_device(ids.data_ptr(), H, offsets.data_ptr(), nodes.data_ptr(), lengths.data_ptr())
    torch.cuda.synchronize()
    del ix
    info = {}
    image = b200.build_image_device(nodes, offsets, bidirectional=True, info=info)
    assert info["positions"] == 2 * H * (L + 1)
    g, want = orc.GBWT.load(image), orc.GBWT.load(img.array)
    assert g.bwt_data() == want.bwt_data()
    assert np.array_equal(g.record_starts(), want.record_starts())
    assert (g.alphabet_offset(), g.alphabet_size(), g.sequences(), g.len()) == \
           (want.alphabet_offset(), want.alphabet_size(), want.sequences(), want.len())


def test_built_index_behaves_like_the_expected_image(b200):
    rng = random.Random(11)
    paths = random_paths(rng, "duplicates") + random_paths(rng, "prefixes")
    want, _ = expected_image(b200, paths)
    seqs = gbb.bidirectional_sequences(paths)
    pats = np.array([s[j:j + 3] for s in seqs for j in range(len(s) - 2)] or [[2, 4, 6]], dtype=np.uint64)
    ids = np.arange(len(seqs), dtype=np.uint64)
    for kw in (dict(), dict(checkpoints=True), dict(locate=True)):
        built, ref = b200.GBWT.build(paths, **kw), b200.GBWT.from_bytes(want, **kw)
        states = built.find_extend(pats)
        assert np.array_equal(states.view(np.uint64), ref.find_extend(pats).view(np.uint64))
        for a, b in zip(built.extract(ids), ref.extract(ids)):
            assert np.array_equal(a, b)
        if kw.get("locate"):
            for a, b in zip(built.locate_states(states), ref.locate_states(states)):
                assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    # node labels on a built bidirectional index
    built, ref = b200.GBWT.build(paths), b200.GBWT.from_bytes(want)
    starts, labels = synth.node_labels((built.alphabet_size() - built.alphabet_offset() - 1) // 2, seed=3)  # GBZ::load's count
    for ix in (built, ref):
        ix.attach_graph(starts, labels)
    for a, b in zip(built.extract_dna(ids, endmarker=ord("$")), ref.extract_dna(ids, endmarker=ord("$"))):
        assert np.array_equal(a, b)


def test_device_variant_on_a_side_stream(b200):
    import torch
    rng = random.Random(3)
    paths = random_paths(rng, "duplicates")
    want, _ = expected_image(b200, paths)
    flat = [x for p in paths for x in p]
    pad = 5
    nodes = torch.tensor([7] * pad + flat + [9], dtype=torch.int64, device="cuda")
    offsets = torch.tensor(np.concatenate([[0], np.cumsum([len(p) for p in paths])]) + pad, dtype=torch.int64, device="cuda")
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        image = b200.build_image_device(nodes, offsets, bidirectional=True, stream=side)
    assert image == want
    assert b200.build_image_device(nodes.data_ptr(), offsets.data_ptr(), n=len(paths), stream=side.cuda_stream) == want


def test_errors(b200):
    import torch
    lib, good = b200.library(), [[2, 4, 6], [4, 6]]

    def host_status(nodes, offsets, n, bidirectional=1):
        image, ln = b200.C.c_void_p(), b200.C.c_size_t(0)
        return lib.gbwt_b200_build_image(nodes, offsets, n, bidirectional, 0, b200.C.byref(image), b200.C.byref(ln), None)

    def code_of(fn, *args, **kw):
        with pytest.raises(b200.GBWTError) as e:
            fn(*args, **kw)
        return e.value.code

    def arrays(nodes, offsets):
        return np.asarray(nodes, dtype=np.uint64), np.asarray(offsets, dtype=np.uint64)

    def both(nodes, offsets, bidirectional=True):
        n, o = arrays(nodes, offsets)
        host = code_of(b200.build_image, (n, o), bidirectional=bidirectional)
        d_n = torch.tensor(n.astype(np.int64), device="cuda")
        d_o = torch.tensor(o.astype(np.int64), device="cuda")
        dev = code_of(b200.build_image_device, d_n, d_o, bidirectional=bidirectional)
        assert host == dev
        return host

    assert code_of(b200.build_image, []) == b200.E_ARGUMENT
    assert code_of(b200.build_image_device, 0, 0, n=0) == b200.E_ARGUMENT
    n, o = arrays([2, 4], [0, 2])
    assert host_status(None, b200._ptr(o), 1) == b200.E_ARGUMENT
    assert host_status(b200._ptr(n), None, 1) == b200.E_ARGUMENT
    d_o = torch.tensor([0, 2], dtype=torch.int64, device="cuda")
    assert code_of(b200.build_image_device, 0, d_o) == b200.E_ARGUMENT
    assert both([2, 4, 6], [0, 2, 1]) == b200.E_ARGUMENT            # offsets decrease
    assert both([2, 0, 6], [0, 3]) == b200.E_ARGUMENT               # node 0
    assert both([2, 1, 6], [0, 3]) == b200.E_ARGUMENT               # node 1: its flip is the endmarker
    assert both([2, U32, 6], [0, 3], bidirectional=False) == b200.E_RANGE
    assert both([2, U32 + 6], [0, 2]) == b200.E_RANGE
    # nodes + sequences >= 2^32: decided from the offsets, before the nodes are read
    assert both([2, 4], [0, U32 // 2]) == b200.E_RANGE
    assert both([2, 4], [0, U32 - 1], bidirectional=False) == b200.E_RANGE
    # the working set does not fit: fill the device but for 1 GiB, then ask for some 2 GiB
    big = np.arange(2, 2 + (48 << 20), dtype=np.int64)
    d_big = torch.tensor(big, device="cuda")
    d_off = torch.tensor([0, len(big)], dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    free, _ = torch.cuda.mem_get_info()
    filler = torch.empty(free - (1 << 30), dtype=torch.uint8, device="cuda")
    with pytest.raises(b200.GBWTError) as e:
        b200.build_image_device(d_big, d_off, bidirectional=False)
    assert e.value.code == b200.E_CUDA and "free" in str(e.value)
    del filler, d_big
    torch.cuda.empty_cache()
    # a failed call leaves nothing behind: the next build on the device succeeds
    assert b200.build_image(good) == expected_image(b200, good)[0]


def test_nothing_stays_allocated(b200):
    import torch
    paths = [[2 * (i % 50) + 2 for i in range(j, j + 200)] for j in range(200)]
    b200.build_image(paths)
    torch.cuda.synchronize()
    before, _ = torch.cuda.mem_get_info()
    for _ in range(3):
        b200.build_image(paths)
    after, _ = torch.cuda.mem_get_info()
    assert after >= before - (2 << 20)


def test_deterministic(b200):
    rng = random.Random(99)
    paths = random_paths(rng, "duplicates") * 3
    assert b200.build_image(paths) == b200.build_image(paths)
    S, H = 2000, 64
    p = chain_paths(S, H, 7)
    assert b200.build_image(p) == b200.build_image(p)
