"""Ranges of sequences on config 4 (10 M nodes x 1024 haplotypes, BASELINE.json configs[3]'s index), one JSON line.

    python tools/bench_ranges.py [--min-seconds 0.5]

Timed with CUDA events on the device entry points (one warm-up, then repeats totalling at least --min-seconds), with the
default path checkpoints:
- seek of 2^24 random (s, j);
- 2^20 node ranges of 64 nodes (locate contexts) and 1024 node ranges of 1 M nodes;
- 2^20 DNA ranges of 1 kbp and 1024 of 1 Mbp, with the synthetic labels of `bench.py --workload extract-dna`;
- whole-path extraction (extract_device / extract_dna_device) of 64 sequences, for the walk rate of the shipped kernels on
  the same card in the same call.
For each: ranges/s, output bytes/s and LF steps/s. The LF steps of a range call are counted from the checkpoint table's
interval: every node written is one step, plus the skip from the checkpoint before the range start (its distance from
the interval's multiple, a lower bound by at most 31 per range); the extraction's steps are its nodes.
Checks: synth.patterns took query q from sequence 2h + o at nodes [t, t + 32), so extract_ranges(2h + o, t, t + 32) must
be the pattern and seek(2h + o, t + 31) its last node; DNA ranges must be slices of extract_dna for a few whole sequences.
Writes nothing into the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

SEED, SEED_Q, K = 42, 7, 32
CONFIG4 = (3_333_333, 1024)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        power = "unknown"
    return name, power


def timed(run, stream, min_seconds):
    """Device milliseconds per call: one warm-up, then repeats totalling at least min_seconds."""
    import torch
    with torch.cuda.stream(stream):
        run()
        stream.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps, ms = 0, 0.0
        while ms < min_seconds * 1e3:
            t0.record(stream)
            run()
            t1.record(stream)
            t1.synchronize()
            ms += t0.elapsed_time(t1)
            reps += 1
    return ms / reps, reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-seconds", type=float, default=0.5)
    args = ap.parse_args()

    import torch
    import gbwt_rs_b200 as gb
    from locate_oracle import pattern_origins
    from synth import synth

    dev = torch.device("cuda", 0)
    name, power = card()
    S, H = CONFIG4
    img = synth.bubble_chain(S, H, SEED)
    for knob in ("GBWT_B200_CHECKPOINTS", "GBWT_B200_CHECKPOINT_SHIFT", "GBWT_B200_DNA_CHECKPOINTS"):
        os.environ.pop(knob, None)
    e = gb.GBWT.from_bytes(img.array, checkpoints=True)
    starts_l, labels = synth.node_labels(3 * S + 1, seed=SEED, max_anchor=32)
    e.attach_graph(starts_l, labels)
    interval = e.checkpoint_info()["interval"]
    n_seq = e.sequences()
    lens = e.sequence_lengths(np.arange(n_seq, dtype=np.uint64))
    dna_lens = e.dna_lengths(np.arange(n_seq, dtype=np.uint64)) - np.uint64(1)
    stream = torch.cuda.Stream(device=dev)
    rng = np.random.default_rng(SEED)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a).astype(np.int64)).to(dev)
    results = {}

    def skip(starts):
        return int(np.sum(starts % np.uint64(interval)))

    # seek
    Q = 1 << 24
    ids = rng.integers(0, n_seq, Q).astype(np.uint64)
    js = (rng.random(Q) * lens[ids]).astype(np.uint64)
    d_ids, d_js, d_out = t(ids), t(js), torch.empty(2 * Q, dtype=torch.int64, device=dev)
    ms, reps = timed(lambda: e.seek_device(d_ids.data_ptr(), d_js.data_ptr(), Q, d_out.data_ptr(), stream.cuda_stream), stream, args.min_seconds)
    steps = skip(js)
    results["seek_2e24"] = {"ms": ms, "passes": reps, "ranges_per_s": Q / (ms / 1e3), "lf_steps_per_s": steps / (ms / 1e3),
                            "output_bytes_per_s": 16 * Q / (ms / 1e3)}
    del d_ids, d_js, d_out

    def ranges(label, m, span, dna):
        full = dna_lens if dna else lens
        ids = rng.integers(0, n_seq, m).astype(np.uint64)
        a = (rng.random(m) * (full[ids] - np.uint64(span))).astype(np.uint64)
        b = a + np.uint64(span)
        width = 1 if dna else 8
        offsets = np.arange(m + 1, dtype=np.uint64) * np.uint64(span)
        d = [t(x) for x in (ids, a, b, offsets)]
        out = torch.empty(m * span * width // 8 + 1, dtype=torch.int64, device=dev)
        d_len = torch.empty(m, dtype=torch.int64, device=dev)
        fn = e.extract_dna_ranges_device if dna else e.extract_ranges_device
        ms, reps = timed(lambda: fn(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), m, d[3].data_ptr(), out.data_ptr(), d_len.data_ptr(),
                                    stream.cuda_stream), stream, args.min_seconds)
        assert bool((d_len == span).all()), label
        nodes = m * span if not dna else None
        results[label] = {"ms": ms, "passes": reps, "ranges_per_s": m / (ms / 1e3), "output_bytes_per_s": m * span * width / (ms / 1e3)}
        if not dna:
            results[label]["lf_steps_per_s"] = (nodes + skip(a)) / (ms / 1e3)
        del out, d

    ranges("node_ranges_2e20_x64", 1 << 20, 64, False)
    ranges("node_ranges_1024_x1M", 1024, 1 << 20, False)
    ranges("dna_ranges_2e20_x1kbp", 1 << 20, 1000, True)
    ranges("dna_ranges_1024_x1Mbp", 1024, 1_000_000, True)

    # whole paths through the shipped kernels, same card, same call
    W = 64
    w_ids = np.arange(W, dtype=np.uint64)
    w_off = np.zeros(W + 1, np.uint64)
    np.cumsum(lens[:W], out=w_off[1:])
    d_w, d_o = t(w_ids), t(w_off)
    out = torch.empty(int(w_off[-1]), dtype=torch.int64, device=dev)
    d_len = torch.empty(W, dtype=torch.int64, device=dev)
    ms, reps = timed(lambda: e.extract_device(d_w.data_ptr(), W, d_o.data_ptr(), out.data_ptr(), d_len.data_ptr(), stream.cuda_stream),
                     stream, args.min_seconds)
    results["extract_64_whole_paths"] = {"ms": ms, "passes": reps, "lf_steps_per_s": int(w_off[-1]) / (ms / 1e3),
                                         "output_bytes_per_s": 8 * int(w_off[-1]) / (ms / 1e3)}
    del out
    dl = e.dna_lengths(w_ids)
    w_doff = np.zeros(W + 1, np.uint64)
    np.cumsum(dl, out=w_doff[1:])
    d_do = t(w_doff)
    out = torch.empty(int(w_doff[-1]) // 8 + 1, dtype=torch.int64, device=dev)
    ms, reps = timed(lambda: e.extract_dna_device(d_w.data_ptr(), W, 0, d_do.data_ptr(), out.data_ptr(), d_len.data_ptr(), stream.cuda_stream),
                     stream, args.min_seconds)
    results["extract_dna_64_whole_paths"] = {"ms": ms, "passes": reps, "lf_steps_per_s": int(w_off[-1]) / (ms / 1e3),
                                             "output_bytes_per_s": int(w_doff[-1]) / (ms / 1e3)}
    del out
    torch.cuda.synchronize()

    # checks at full size
    n = 1 << 20
    pats = synth.patterns(S, H, SEED, n=n, k=K, seed_q=SEED_Q)
    seqs, last = pattern_origins(S, H, n, k=K, seed_q=SEED_Q)
    first = last - np.uint64(K - 1)
    _, nodes, _ = e.extract_ranges(seqs, first, first + np.uint64(K))
    patterns_ok = bool(np.array_equal(nodes.reshape(n, K), pats))
    seek_ok = bool(np.array_equal(e.seek(seqs, last)["node"], pats[:, -1]))
    few = np.array([0, 1, 777, n_seq - 1], np.uint64)
    off, whole, _ = e.extract_dna(few)
    a = np.array([0, 12345, 999_999, 5_000_000], np.uint64)
    b = a + np.array([1000, 1_000_000, 3, 4_000_000], np.uint64)
    _, got, _ = e.extract_dna_ranges(few, a, b)
    want = np.concatenate([whole[int(off[i]) + int(a[i]):int(off[i]) + min(int(b[i]), int(off[i + 1] - off[i]) - 1)] for i in range(len(few))])
    dna_ok = bool(np.array_equal(got, want))

    line = {
        "metric": "gbwt_node_ranges_per_s", "value": results["node_ranges_2e20_x64"]["ranges_per_s"], "unit": "ranges/s",
        "card": name, "power_limit": power,
        "config": f"synthetic bubble-chain GBWT, {3 * S + 1} nodes x {H} haplotypes (seed {SEED}), path checkpoints every {interval} "
                  f"nodes, node labels of bench.py --workload extract-dna",
        "results": results,
        "checks": {"pattern_ranges_2e20": patterns_ok, "pattern_last_node_seek_2e20": seek_ok, "dna_ranges_vs_extract_dna": dna_ok},
    }
    print(json.dumps(line))
    if not (patterns_ok and seek_ok and dna_ok):
        sys.exit(1)


if __name__ == "__main__":
    main()
