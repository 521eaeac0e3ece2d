"""The document array of the oracle (tests/locate_oracle.py), which locate is checked against, checked on its own: on
every fixture and on random graphs whose paths visit nodes more than once, it is a bijection between the non-endmarker
positions and the pairs (s, j), j < len(sequence s); start(s) is (s, 0); forward takes (s, j) to (s, j + 1). CPU only."""
import os
import random

import numpy as np
import pytest

import gbwt_builder as gb
from locate_oracle import NONE, DocumentArray
from oracle import oracle as orc
from synth import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FIXTURES = ["example.gbwt", "with-empty.gbwt", "translation.gbwt", "example.gbz", "translation.gbz"]


def image_of(b, bidirectional=True):
    flags = 4 | (1 if bidirectional else 0)
    return synth.gbwt_image(b["sequences"], b["size"], b["offset"], b["alphabet_size"], flags, b["starts"], b["data"])


def random_graph(seed, bidirectional=True):
    """Random walks over few nodes: nodes revisited within a path, high outdegrees, empty paths."""
    rng = random.Random(seed)
    n_nodes = rng.choice([2, 3, 6, 12])
    paths = []
    for _ in range(rng.choice([3, 10, 40])):
        paths.append([2 * rng.randint(1, n_nodes) + (1 if rng.random() < 0.2 else 0) for _ in range(rng.randint(0, rng.choice([3, 8, 20])))])
    if not any(paths):
        paths.append([2, 4, 2])
    seqs = gb.bidirectional_sequences(paths) if bidirectional else paths
    return image_of(gb.build_bwt(seqs), bidirectional), paths


def check_document_array(g):
    da = DocumentArray(g)
    assert da.ok, "a walk visited a position twice or left the records"
    lengths = [len(g.sequence(s)) for s in range(g.sequences())]
    # bijection: every slot is visited (da_build already refused a second visit), and the pairs are exactly {(s, j)}
    assert not np.any(da.seq == NONE)
    assert len(da.seq) == sum(lengths)
    pairs = sorted(zip(da.seq.tolist(), da.idx.tolist()))
    assert pairs == [(s, j) for s in range(g.sequences()) for j in range(lengths[s])]
    positions = da.positions()
    # start(s) -> (s, 0)
    for s in range(g.sequences()):
        p = g.start(s)
        if lengths[s] == 0:
            assert p is None
            continue
        occ = da.locate_batch(np.array([p], orc.POS_DTYPE))[0]
        assert (int(occ["sequence"]), int(occ["index"])) == (s, 0)
    # forward: (s, j) -> (s, j + 1), None after the last node
    for k, pos in enumerate(positions):
        nxt = g.forward((int(pos["node"]), int(pos["offset"])))
        s, j = int(da.seq[k]), int(da.idx[k])
        if nxt is None:
            assert j == lengths[s] - 1
        else:
            occ = da.locate_batch(np.array([nxt], orc.POS_DTYPE))[0]
            assert (int(occ["sequence"]), int(occ["index"])) == (s, j + 1)
    # positions that do not exist
    bad = np.array([(0, 0), (g.first_node() - 1 if g.first_node() > 0 else 0, 0), (g.alphabet_size(), 0), (g.first_node(), 2**40)],
                   orc.POS_DTYPE)
    assert np.all(da.locate_batch(bad)["sequence"] == NONE)
    return da


@pytest.mark.parametrize("name", FIXTURES)
def test_fixtures(name):
    g = orc.GBWT.load(open(os.path.join(GOLDEN, name), "rb").read())
    da = check_document_array(g)
    if name == "with-empty.gbwt":
        assert any(g.start(s) is None for s in range(g.sequences()))  # the empty paths are there, and own no position


@pytest.mark.parametrize("bidirectional", [True, False])
@pytest.mark.parametrize("seed", range(6))
def test_random_graphs(seed, bidirectional):
    img, paths = random_graph(seed, bidirectional)
    g = orc.GBWT.load(img)
    assert any(len(set(p)) < len(p) for p in paths)  # some path visits a node more than once
    check_document_array(g)
