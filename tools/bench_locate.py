"""Locate on config 4 (10 M nodes x 1024 haplotypes, BASELINE.json configs[3]'s index), one JSON line.

    python tools/bench_locate.py [--queries 16777216] [--min-seconds 0.5] [--no-extract]

- Creation: index-ready time with and without GBWT_B200_LAYOUT_LOCATE, and the bytes of the samples.
- Timed run: 2^24 device-synthesised 32-node patterns (synth.patterns_device) go through find_extend_device; then
  locate_states_device on the resulting states is timed with CUDA events (one warm-up, then repeats totalling at least
  --min-seconds): occurrences/s. A separate pass with GBWT_B200_LOCATE_STATS=1 counts the LF steps the walks take, so
  LF steps/s = steps per pass / time per pass of the timed run.
- The same call runs `bench.py --workload extract` for its LF steps/s, so that the two walk rates come from one card.
- Checks: every query's occurrences contain (2h + o, t + 31), where synth.patterns took the query from sequence 2h + o at
  node t; and on config 3 (configs[2]), 2^20 random positions match the oracle's document array.
Writes nothing into the tree (the helper libraries are compiled into temporary directories).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

SEED, SEED_Q, K = 42, 7, 32
CONFIG4 = (3_333_333, 1024)
CONFIG3 = (33_333, 64)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        power = "unknown"
    return name, power


def ready_seconds(gb, image, locate):
    import torch
    torch.cuda.synchronize()
    t = time.perf_counter()
    e = gb.GBWT.from_bytes(image, locate=locate)
    torch.cuda.synchronize()
    return e, time.perf_counter() - t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=1 << 24)
    ap.add_argument("--min-seconds", type=float, default=0.5)
    ap.add_argument("--check-chunk", type=int, default=1 << 20)
    ap.add_argument("--no-extract", action="store_true")
    args = ap.parse_args()

    import torch
    import gbwt_rs_b200 as gb
    from locate_oracle import DocumentArray, pattern_origins
    from oracle import oracle as orc
    from synth import synth

    dev = torch.device("cuda", 0)
    name, power = card()
    S, H = CONFIG4
    img = synth.bubble_chain(S, H, SEED)
    os.environ.pop("GBWT_B200_LOCATE_SHIFT", None)
    os.environ.pop("GBWT_B200_LOCATE_STATS", None)
    plain, plain_s = ready_seconds(gb, img.array, False)
    plain_bytes = plain.device_bytes()["total"]
    del plain
    e, locate_s = ready_seconds(gb, img.array, True)
    info = e.locate_info()

    # queries: find/extend on the device, then the occurrences of the states they reach
    Q = args.queries
    stream = torch.cuda.Stream(device=dev)
    d_pat = torch.empty(Q * K, dtype=torch.int64, device=dev)
    d_states = torch.empty(Q * 3, dtype=torch.int64, device=dev)
    with torch.cuda.stream(stream):
        synth.patterns_device(S, H, SEED, Q, d_pat.data_ptr(), k=K, seed_q=SEED_Q, q0=0, stream=stream.cuda_stream)
        e.find_extend_device(d_pat.data_ptr(), Q, K, d_states.data_ptr(), stream.cuda_stream)
    stream.synchronize()
    del d_pat
    st = d_states.view(Q, 3)
    counts = (st[:, 2] - st[:, 1]).clamp(min=0)
    d_offsets = torch.zeros(Q + 1, dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=d_offsets[1:])
    total = int(d_offsets[-1])
    d_out = torch.empty(2 * total, dtype=torch.int64, device=dev)
    d_counts = torch.empty(Q, dtype=torch.int64, device=dev)

    def run():
        e.locate_states_device(d_states.data_ptr(), Q, d_offsets.data_ptr(), d_out.data_ptr(), d_counts.data_ptr(), stream.cuda_stream)

    with torch.cuda.stream(stream):
        run()  # warm-up
        stream.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps, ms = 0, 0.0
        while ms < args.min_seconds * 1e3:
            t0.record(stream)
            run()
            t1.record(stream)
            t1.synchronize()
            ms += t0.elapsed_time(t1)
            reps += 1
    per_pass_ms = ms / reps
    # LF steps: one more pass with the counter on (its own time is not used)
    os.environ["GBWT_B200_LOCATE_STATS"] = "1"
    before = e.locate_info()["lf_steps"]
    with torch.cuda.stream(stream):
        run()
    stream.synchronize()
    steps = e.locate_info()["lf_steps"] - before
    os.environ.pop("GBWT_B200_LOCATE_STATS")

    # check: every query's occurrences contain (2h + o, t + 31)
    assert torch.equal(d_counts, counts), "counts differ from end - start"
    seqs, idxs = pattern_origins(S, H, Q, k=K, seed_q=SEED_Q)
    d_seqs = torch.from_numpy(seqs.astype(np.int64)).to(dev)
    d_idxs = torch.from_numpy(idxs.astype(np.int64)).to(dev)
    occ = d_out.view(total, 2)
    missing = 0
    for q0 in range(0, Q, args.check_chunk):
        q1 = min(Q, q0 + args.check_chunk)
        lo, hi = int(d_offsets[q0]), int(d_offsets[q1])
        owner = torch.repeat_interleave(torch.arange(q0, q1, device=dev), counts[q0:q1])
        hit = (occ[lo:hi, 0] == d_seqs[owner]) & (occ[lo:hi, 1] == d_idxs[owner])
        found = torch.zeros(q1 - q0, dtype=torch.int64, device=dev).index_add_(0, owner - q0, hit.to(torch.int64))
        missing += int((found != 1).sum())
    del e, d_out, d_states

    # check: config 3 against the oracle's document array
    S3, H3 = CONFIG3
    img3 = synth.bubble_chain(S3, H3, SEED)
    g3 = orc.GBWT.load(img3.array)
    da = DocumentArray(g3)
    e3 = gb.GBWT.from_bytes(img3.array, locate=True)
    rng = np.random.default_rng(SEED)
    positions = da.positions()[rng.integers(0, len(da.seq), 1 << 20)]
    config3_ok = bool(np.array_equal(e3.locate_positions(positions).view(np.uint64), da.locate_batch(positions).view(np.uint64)))

    extract = None
    if not args.no_extract:
        proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "extract", "--gpus", "1", "--steps", "3",
                               "--warmup", "1"], capture_output=True, text=True)
        lines = [ln for ln in proc.stdout.splitlines() if ln.startswith("{")]
        extract = json.loads(lines[-1])["value"] if proc.returncode == 0 and lines else f"failed ({proc.returncode})"

    line = {
        "metric": "gbwt_locate_occurrences_per_s", "value": total / (per_pass_ms / 1e3), "unit": "occurrences/s",
        "card": name, "power_limit": power,
        "config": f"synthetic bubble-chain GBWT, {3 * S + 1} nodes x {H} haplotypes (seed {SEED}), {Q} length-{K} patterns "
                  f"(seed {SEED_Q}) through find_extend_device, then locate_states_device; samples every {info['interval']} nodes",
        "queries": Q, "occurrences": total, "ms_per_pass": per_pass_ms, "timed_passes": reps,
        "lf_steps_per_pass": steps, "locate_lf_steps_per_s": steps / (per_pass_ms / 1e3),
        "extract_lf_steps_per_s": extract,
        "index_ready_s": {"without_samples": plain_s, "with_samples": locate_s},
        "samples": info["samples"], "sample_bytes": info["bytes"], "sample_build_us": info["build_us"],
        "device_bytes": {"without_samples": plain_bytes, "with_samples": plain_bytes + info["bytes"]},
        "checks": {"queries_missing_their_origin": missing, "config3_oracle_2e20_positions": config3_ok},
    }
    print(json.dumps(line))
    if missing or not config3_ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
