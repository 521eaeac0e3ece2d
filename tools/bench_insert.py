"""Inserting haplotype paths into a loaded GBWT (GBWT.insert_image_device) on bubble chains, one JSON line per insert.

    python tools/bench_insert.py [--sites 3333333] [--haplotypes 128] [--first 64] [--step 64]

The first `--first` haplotypes of the chain are built on the device and loaded; then the rest are inserted `--step` at a time,
each result loaded with GBWT.from_bytes before the next insert. Per insert: the wall time of the blocking call, its device
time split from the kernel trace of torch.profiler into S's build (S's sort and A's incoming-edge table, before the walk),
the insertion walk, and the record pass (S's entries and edges, the merged edges and records); the host time of the file
write (wall minus device) and of from_bytes; peak device bytes next to the memory rule (36 B per new position, 36 B per edge
of A, the output). The final image is checked against the synth image of the whole chain. `--sites 3333333
--haplotypes 1024 --first 128 --step 128` is config 4 built in eight pieces. Writes nothing into the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

from bench_build import SEED, card  # noqa: E402


def device_split(call):
    """Device microseconds of the kernels before k_insert_walk, of the walk, and after it, for one call."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "Memcpy" not in e.name
                      and "Memset" not in e.name), key=lambda e: e.time_range.start)
    parts = [0.0, 0.0, 0.0]
    phase = 0
    for e in kernels:
        if "k_insert_walk" in e.name:
            phase = 1
        elif phase == 1:
            phase = 2
        parts[phase] += e.time_range.elapsed_us()
    return parts


def paths_on_device(S, H, h0, h1):
    import torch
    from synth import synth
    L = 2 * S + 1
    nodes = np.empty((h1 - h0) * L, dtype=np.int64)
    for h in range(h0, h1):
        nodes[(h - h0) * L:(h - h0 + 1) * L] = synth.sequence(S, H, SEED, 2 * h).astype(np.int64)
    return torch.from_numpy(nodes).cuda(), torch.arange(0, h1 - h0 + 1, dtype=torch.int64, device="cuda") * L


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=3_333_333)
    ap.add_argument("--haplotypes", type=int, default=128)
    ap.add_argument("--first", type=int, default=64)
    ap.add_argument("--step", type=int, default=64)
    ap.add_argument("--profile", type=int, default=1, help="split the device time of each insert with torch.profiler (one more run)")
    args = ap.parse_args()
    import torch
    import gbwt_rs_b200 as gb
    from oracle import oracle as orc
    from synth import synth
    name, power = card()
    S, H = args.sites, args.haplotypes
    d_nodes, d_offsets = paths_on_device(S, H, 0, args.first)
    t0 = time.perf_counter()
    image = gb.build_image_device(d_nodes, d_offsets, bidirectional=True)
    build_s = time.perf_counter() - t0
    del d_nodes, d_offsets
    torch.cuda.empty_cache()
    t0 = time.perf_counter()
    ix = gb.GBWT.from_bytes(image)
    print(json.dumps(dict(step="build", sites=S, haplotypes=args.first, build_s=round(build_s, 3),
                          from_bytes_host_s=round(time.perf_counter() - t0, 3), card=name, power_limit=power)), flush=True)
    h = args.first
    while h < H:
        h1 = min(H, h + args.step)
        d_nodes, d_offsets = paths_on_device(S, H, h, h1)
        info = {}
        t0 = time.perf_counter()
        image = ix.insert_image_device(d_nodes, d_offsets, info=info)
        wall = time.perf_counter() - t0
        split = device_split(lambda: ix.insert_image_device(d_nodes, d_offsets)) if args.profile else [0.0, 0.0, 0.0]
        a_edge_lists = ix.device_bytes()["edges"]
        del d_nodes, d_offsets, ix
        torch.cuda.empty_cache()
        t0 = time.perf_counter()
        ix = gb.GBWT.from_bytes(image)
        from_bytes_s = time.perf_counter() - t0
        print(json.dumps(dict(step="insert", sites=S, haplotypes_before=h, inserted=h1 - h, positions=info["positions"],
                              rounds=info["rounds"], wall_s=round(wall, 3), device_us=info["device_us"], walk_us=info["walk_us"],
                              longest=info["longest"], s_build_kernel_us=round(split[0]), walk_kernel_us=round(split[1]),
                              record_pass_kernel_us=round(split[2]), host_write_s=round(wall - info["device_us"] / 1e6, 3),
                              from_bytes_host_s=round(from_bytes_s, 3), peak_device_bytes=info["peak_device_bytes"],
                              rule_36b_per_new_position=36 * info["positions"], a_edge_list_bytes=a_edge_lists, image_bytes=len(image),
                              card=name, power_limit=power)), flush=True)
        h = h1
    del ix
    chain = synth.bubble_chain(S, H, SEED)  # kept alive: the oracle reads its array in place
    want = orc.GBWT.load(chain.array)
    g = orc.GBWT.load(image)
    ok = g.bwt_data() == want.bwt_data() and np.array_equal(g.record_starts(), want.record_starts()) and \
        (g.alphabet_offset(), g.alphabet_size(), g.sequences(), g.len()) == (want.alphabet_offset(), want.alphabet_size(), want.sequences(), want.len())
    print(json.dumps(dict(step="check", sites=S, haplotypes=H, matches_synth=bool(ok))), flush=True)
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
