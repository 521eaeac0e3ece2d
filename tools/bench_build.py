"""Building a GBWT from paths on the device (gbwt_b200_build_image_device) on bubble chains, one JSON line per size.

    python tools/bench_build.py [--sizes 33333x64,3333333x128] [--repeats 3]

For each size the forward paths of synth.sequence are copied to the device once; then one warm-up build and --repeats timed
builds (host clock around the blocking call, which ends with the image on the host). Reported: positions/s (nodes +
sequences), the doubling rounds, the peak device bytes, and, from one extra build under torch.profiler, the device time of
the kernels up to the first record kernel (k_build_entries: symbol sort and doubling rounds) and after it (records, edges,
runs, encoding). Also the host time of GBWT.from_bytes on the built image (the existing host layout pass). Every built image
is checked against the synth image of the same chain: BWT bytes, record starts and header through the oracle.
Writes nothing into the tree.
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
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

SEED = 42


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        power = "unknown"
    return name, power


def device_split(build):
    """Device microseconds of the kernels before the first k_build_entries and from it on, for one build."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        build()
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "Memcpy" not in e.name
                      and "Memset" not in e.name), key=lambda e: e.time_range.start)
    doubling = records = 0.0
    seen = False
    for e in kernels:
        seen = seen or "k_build_entries" in e.name
        if seen:
            records += e.time_range.elapsed_us()
        else:
            doubling += e.time_range.elapsed_us()
    return doubling, records


def run(S: int, H: int, repeats: int) -> dict:
    import torch
    import gbwt_rs_b200 as gb
    from oracle import oracle as orc
    from synth import synth
    L = 2 * S + 1
    nodes = np.empty(H * L, dtype=np.int64)
    for h in range(H):
        nodes[h * L:(h + 1) * L] = synth.sequence(S, H, SEED, 2 * h).astype(np.int64)
    d_nodes = torch.from_numpy(nodes).cuda()
    d_offsets = torch.arange(0, H + 1, dtype=torch.int64, device="cuda") * L
    del nodes
    info = {}
    build = lambda: gb.build_image_device(d_nodes, d_offsets, bidirectional=True, info=info)
    image = build()
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        again = build()
        times.append(time.perf_counter() - t0)
        assert again == image
    doubling_us, records_us = device_split(build)
    del d_nodes, d_offsets
    torch.cuda.empty_cache()
    t0 = time.perf_counter()
    ix = gb.GBWT.from_bytes(image)
    from_bytes_s = time.perf_counter() - t0
    del ix
    want = synth.bubble_chain(S, H, SEED)
    g, w = orc.GBWT.load(image), orc.GBWT.load(want.array)
    ok = g.bwt_data() == w.bwt_data() and np.array_equal(g.record_starts(), w.record_starts()) and \
        (g.alphabet_offset(), g.alphabet_size(), g.sequences(), g.len()) == (w.alphabet_offset(), w.alphabet_size(), w.sequences(), w.len())
    best = min(times)
    return dict(sites=S, haplotypes=H, positions=info["positions"], rounds=info["rounds"], build_s=round(best, 4),
                build_s_all=[round(t, 4) for t in times], positions_per_s=round(info["positions"] / best),
                device_us_reported=info["device_us"], doubling_kernel_us=round(doubling_us), records_kernel_us=round(records_us),
                peak_device_bytes=info["peak_device_bytes"], image_bytes=len(image), from_bytes_host_s=round(from_bytes_s, 3),
                matches_synth=bool(ok))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="33333x64,3333333x128")
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    name, power = card()
    for size in args.sizes.split(","):
        S, H = (int(x) for x in size.split("x"))
        row = run(S, H, args.repeats)
        row.update(card=name, power_limit=power)
        print(json.dumps(row), flush=True)
        if not row["matches_synth"]:
            sys.exit(1)


if __name__ == "__main__":
    main()
