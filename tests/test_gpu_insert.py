"""Inserting paths into a loaded GBWT on the GPU (gbwt_b200_insert_image, include/gbwt_b200_insert.h).

The image must be byte for byte both what from_parts(<tests/gbwt_builder.py of seqs(A) + S>).serialize() writes and
build_image(paths(A) + P) with A's orientation, for A loaded in every body layout, and the loaded result must answer like
the build of the same paths."""
import os
import random

import numpy as np
import pytest

import gbwt_builder as gbb
from oracle import oracle as orc
from synth import synth
from test_gpu_build import U32, chain_paths, random_paths

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LOADS = [dict(), dict(layout="runs"), dict(checkpoints=True), dict(layout="runs", checkpoints=False, locate=True)]


@pytest.fixture(scope="module")
def b200():
    import gbwt_rs_b200
    return gbwt_rs_b200


def a_paths(g):
    seqs = [[int(x) for x in g.sequence(i)] for i in range(g.sequences())]
    return seqs[0::2] if g.is_bidirectional() else seqs


def expected(b200, paths, bidirectional):
    b = gbb.build_bwt(gbb.bidirectional_sequences(paths) if bidirectional else [list(p) for p in paths])
    ix = b200.GBWT.from_parts(b["sequences"], b["size"], b["offset"], b["alphabet_size"], 1 if bidirectional else 0, b["data"], b["starts"])
    return ix.serialize()


def check_insert(b200, a, old, new, bidirectional):
    info = {}
    image = a.insert_image(new, info=info)
    want = b200.build_image(old + new, bidirectional=bidirectional)
    assert image == want
    assert image == expected(b200, old + new, bidirectional)
    assert info["peak_device_bytes"] > 0 and info["longest"] == max([len(p) for p in new] + [0])
    return image


def new_paths(rng, old, lo, hi):
    walk = lambda n: [2 * rng.randint(lo, hi) + (1 if rng.random() < 0.3 else 0) for _ in range(n)]
    out = [walk(rng.randint(1, 8)) for _ in range(rng.randint(1, 6))]
    if old:
        p = list(rng.choice(old))
        out += [p, p, p[:rng.randint(0, len(p))], p + walk(3), walk(2) + p]
    out += [[], [2 * hi + 2], [max(2, 2 * lo - 2)], [2 * hi + 6, 2 * lo, 2 * hi + 6]]
    rng.shuffle(out)
    return out


@pytest.mark.parametrize("name", ["example.gbwt", "with-empty.gbwt", "translation.gbwt", "example.gbz"])
@pytest.mark.parametrize("load", range(len(LOADS)))
def test_fixtures(b200, name, load):
    path = os.path.join(GOLDEN, name)
    g = orc.GBWT.load(path)
    old = a_paths(g)
    nodes = [x // 2 for p in old for x in p]
    a = b200.GBWT.load(path, **LOADS[load])
    before = a.serialize()
    rng = random.Random(f"{name}-{load}")
    for _ in range(3):
        check_insert(b200, a, old, new_paths(rng, old, max(1, min(nodes) - 2), max(nodes) + 2), True)
    assert a.serialize() == before


@pytest.mark.parametrize("bidirectional", [True, False])
@pytest.mark.parametrize("kind", ["plain", "duplicates", "prefixes", "short", "wide", "long_runs", "sparse", "high"])
def test_random_paths(b200, kind, bidirectional):
    rng = random.Random(f"insert-{kind}-{bidirectional}")
    for t in range(4):
        old = random_paths(rng, kind)
        # "plain" paths next to A's "sparse" ones: new nodes below and between A's; "high" stays high (ids near 2^32)
        new = random_paths(rng, kind if t % 2 or kind == "high" else "plain")
        while kind == "high" and any(x < U32 // 2 for p in old + new for x in p):
            # random_paths adds [2, 4, 2] to a set of empty paths: next to high ids that spans 2^32 records, which the
            # brute-force builder cannot write
            old, new = random_paths(rng, kind), random_paths(rng, kind)
        a = b200.GBWT.build(old, bidirectional=bidirectional, **LOADS[t % len(LOADS)])
        check_insert(b200, a, old, new, bidirectional)


def test_runs_split_and_joined(b200):
    """S entries inside one of A's runs split it; S entries between two runs of one value join them."""
    old = [[2, 4, 8]] * 20 + [[2, 6, 8]] * 20 + [[2, 4, 8]] * 20
    for new in ([[2, 6, 8]], [[2, 4, 8]] * 3, [[2, 6, 8], [2, 4, 8]] * 30, [[2, 4, 10]], [[4, 8]] * 300):
        for load in LOADS:
            check_insert(b200, b200.GBWT.build(old, **load), old, new, True)


def test_outdegree_crosses_255(b200):
    old = [[4, 2 * k] for k in range(3, 3 + 250)]
    new = [[4, 2 * k] for k in range(300, 320)] + [[4, 6]] * 3
    for load in LOADS:
        check_insert(b200, b200.GBWT.build(old, **load), old, new, True)


def test_chained_inserts(b200):
    rng = random.Random(5)
    for bidirectional in (True, False):
        p0, p1, p2 = (random_paths(rng, "duplicates") for _ in range(3))
        a = b200.GBWT.build(p0, bidirectional=bidirectional)
        b = a.insert(p1, layout="runs")
        image = b.insert_image(p2)
        assert image == b200.build_image(p0 + p1 + p2, bidirectional=bidirectional)


@pytest.mark.parametrize("S,H,seed,kw", [(500, 64, 42, {}), (3000, 100, 9, dict(alt_ppm=200_000, tri_mod=3))])
def test_bubble_chain_in_pieces(b200, S, H, seed, kw):
    paths = chain_paths(S, H, seed, **kw)
    img = synth.bubble_chain(S, H, seed, **kw)  # kept alive: the oracle reads its array in place
    want = orc.GBWT.load(img.array)
    q = H // 4
    ix = b200.GBWT.build(paths[:q])
    for k in range(1, 4):
        end = (k + 1) * q if k < 3 else H
        image = ix.insert_image(paths[k * q:end])
        assert image == b200.build_image(paths[:end]), k
        ix = b200.GBWT.from_bytes(image)
    g = orc.GBWT.load(image)
    assert g.bwt_data() == want.bwt_data()
    assert np.array_equal(g.record_starts(), want.record_starts())


def test_inserted_index_behaves_like_the_build(b200):
    rng = random.Random(11)
    old, new = random_paths(rng, "duplicates"), random_paths(rng, "prefixes")
    seqs = gbb.bidirectional_sequences(old + new)
    pats = np.array([s[j:j + 3] for s in seqs for j in range(len(s) - 2)] or [[2, 4, 6]], dtype=np.uint64)
    ids = np.arange(len(seqs), dtype=np.uint64)
    a = b200.GBWT.build(old)
    for kw in (dict(), dict(checkpoints=True), dict(locate=True)):
        got, ref = a.insert(new, **kw), b200.GBWT.build(old + new, **kw)
        states = got.find_extend(pats)
        assert np.array_equal(states.view(np.uint64), ref.find_extend(pats).view(np.uint64))
        for x, y in zip(got.extract(ids), ref.extract(ids)):
            assert np.array_equal(x, y)
        if kw.get("locate"):
            for x, y in zip(got.locate_states(states), ref.locate_states(states)):
                assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
        if kw.get("checkpoints"):
            starts, ends = np.ones(len(ids), np.uint64), np.full(len(ids), 4, np.uint64)
            for x, y in zip(got.extract_ranges(ids, starts, ends), ref.extract_ranges(ids, starts, ends)):
                assert np.array_equal(x, y)


def test_merge_two_indexes_through_extract_device(b200):
    import torch
    rng = random.Random(21)
    pa, pb = random_paths(rng, "plain"), random_paths(rng, "duplicates")
    a, b = b200.GBWT.build(pa), b200.GBWT.build(pb)
    n = len(pb)
    lengths = [len(p) for p in pb]
    ids = torch.arange(0, 2 * n, 2, dtype=torch.int64, device="cuda")
    offsets = torch.tensor(np.concatenate([[0], np.cumsum(lengths)]), dtype=torch.int64, device="cuda")
    nodes = torch.empty(max(sum(lengths), 1), dtype=torch.int64, device="cuda")
    out_len = torch.empty(n, dtype=torch.int64, device="cuda")
    b.extract_device(ids.data_ptr(), n, offsets.data_ptr(), nodes.data_ptr(), out_len.data_ptr())
    torch.cuda.synchronize()
    assert a.insert_image_device(nodes, offsets) == b200.build_image(pa + pb)


def test_device_variant_on_a_side_stream(b200):
    import torch
    rng = random.Random(3)
    old, new = random_paths(rng, "duplicates"), random_paths(rng, "short")
    a = b200.GBWT.build(old)
    want = b200.build_image(old + new)
    flat = [x for p in new for x in p]
    pad = 5
    nodes = torch.tensor([7] * pad + flat + [9], dtype=torch.int64, device="cuda")
    offsets = torch.tensor(np.concatenate([[0], np.cumsum([len(p) for p in new])]) + pad, dtype=torch.int64, device="cuda")
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        image = a.insert_image_device(nodes, offsets, stream=side)
    assert image == want
    assert a.insert_image_device(nodes.data_ptr(), offsets.data_ptr(), n=len(new), stream=side.cuda_stream) == want


def test_errors(b200):
    import torch
    lib = b200.library()
    good_old, good_new = [[2, 4, 6], [4, 6]], [[6, 8]]
    a = b200.GBWT.build(good_old)
    u = b200.GBWT.build(good_old, bidirectional=False)

    def code_of(fn, *args, **kw):
        with pytest.raises(b200.GBWTError) as e:
            fn(*args, **kw)
        return e.value.code

    def both(ix, nodes, offsets):
        n, o = np.asarray(nodes, dtype=np.uint64), np.asarray(offsets, dtype=np.uint64)
        host = code_of(ix.insert_image, (n, o))
        dev = code_of(ix.insert_image_device, torch.tensor(n.astype(np.int64), device="cuda"), torch.tensor(o.astype(np.int64), device="cuda"))
        assert host == dev
        return host

    image, ln = b200.C.c_void_p(), b200.C.c_size_t(0)
    n, o = np.asarray([2, 4], np.uint64), np.asarray([0, 2], np.uint64)
    assert lib.gbwt_b200_insert_image(None, b200._ptr(n), b200._ptr(o), 1, b200.C.byref(image), b200.C.byref(ln), None) == b200.E_ARGUMENT
    assert lib.gbwt_b200_insert_image(a._h, b200._ptr(n), None, 1, b200.C.byref(image), b200.C.byref(ln), None) == b200.E_ARGUMENT
    assert lib.gbwt_b200_insert_image(a._h, None, b200._ptr(o), 1, b200.C.byref(image), b200.C.byref(ln), None) == b200.E_ARGUMENT
    assert code_of(a.insert_image, []) == b200.E_ARGUMENT
    assert both(a, [2, 4, 6], [0, 2, 1]) == b200.E_ARGUMENT     # offsets decrease
    assert both(a, [2, 0, 6], [0, 3]) == b200.E_ARGUMENT        # node 0
    assert both(a, [2, 1, 6], [0, 3]) == b200.E_ARGUMENT        # node 1 into a bidirectional index
    assert u.insert_image([[1, 2]]) == b200.build_image(good_old + [[1, 2]], bidirectional=False)
    assert both(u, [2, U32, 6], [0, 3]) == b200.E_RANGE
    assert both(a, [2, 4], [0, U32 // 2]) == b200.E_RANGE       # new nodes + sequences >= 2^32
    # the working set does not fit
    big = np.arange(2, 2 + (48 << 20), dtype=np.int64)
    d_big = torch.tensor(big, device="cuda")
    d_off = torch.tensor([0, len(big)], dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    free, _ = torch.cuda.mem_get_info()
    filler = torch.empty(free - (1 << 30), dtype=torch.uint8, device="cuda")
    with pytest.raises(b200.GBWTError) as e:
        u.insert_image_device(d_big, d_off)
    assert e.value.code == b200.E_CUDA and "free" in str(e.value)
    del filler, d_big
    torch.cuda.empty_cache()
    assert a.insert_image(good_new) == b200.build_image(good_old + good_new)


def test_a_unchanged_nothing_left_deterministic(b200):
    import torch
    rng = random.Random(99)
    old = [[2 * (i % 50) + 2 for i in range(j, j + 200)] for j in range(100)]
    new = random_paths(rng, "duplicates") * 3
    a = b200.GBWT.build(old, locate=True)
    before = a.serialize()
    pats = np.array([[2, 4, 6], [10, 12, 14], [100, 2, 4]], dtype=np.uint64)
    states = a.find_extend(pats)
    first = a.insert_image(new)
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    for _ in range(3):
        assert a.insert_image(new) == first
    free1, _ = torch.cuda.mem_get_info()
    assert free1 >= free0 - (2 << 20)
    assert a.serialize() == before
    assert np.array_equal(a.find_extend(pats).view(np.uint64), states.view(np.uint64))
