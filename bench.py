#!/usr/bin/env python
"""bench.py -- headline benchmark: batched GBWT find/extend queries per second (k = 32) on B200.

    python bench.py [--gpus N --steps K --warmup W]                      (N = 1)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...       the CPU restatement of the reference path on the host cores

Workload (BASELINE.json configs[3]): synthetic chromosome-scale bubble-chain GBWT, 10 M nodes x 1024
haplotypes (3 333 333 sites), length-32 patterns sampled from the haplotypes (SURVEY.md 8(d)); the index is
replicated on every GPU and the queries are sharded (weak scaling: 2^26 queries per GPU per step, ~1.07 G
queries per step at 8 GPUs). A step is one pass of the hot path over the rank's batch. One JSON line on stdout.

Other workloads for development: --workload find-c3 (configs[2]), --workload extract (configs[4]).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from, which may be read-only

WORKLOADS = {
    # name: (sites, haplotypes, queries per GPU per step)
    "find": (3_333_333, 1024, 1 << 26),
    "find-c3": (33_333, 64, 10_000_000),
    "extract": (3_333_333, 1024, 0),
    "extract-dna": (3_333_333, 1024, 0),
    # the run-length workload: 10 M node ids x 1024 haplotypes with alternative alleles of frequency 0.05 and every tenth
    # site tri-allelic (synth variant model): anchors with three edges keep run-length bodies (records_run8 > 0)
    "find-runs": (2_500_000, 1024, 1 << 26),
}
SEED, SEED_Q, K_LEN = 42, 7, 32
# allele model per workload (synth.bubble_chain): alt_ppm = 0 is the default model (two equally likely alleles)
MODELS = {"find-runs": {"alt_ppm": 50_000, "tri_mod": 10}}


def model_of(args):
    return MODELS.get(args.workload, {"alt_ppm": 0, "tri_mod": 0})


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="find")
    ap.add_argument("--sites", type=int, default=0, help="override the number of sites (development only)")
    ap.add_argument("--haplotypes", type=int, default=0)
    ap.add_argument("--queries", type=int, default=0, help="queries per GPU per step")
    ap.add_argument("--e2e-queries", type=int, default=1 << 24, help="queries per GPU per end-to-end step")
    ap.add_argument("--layout", choices=["auto", "runs"], default="auto")
    ap.add_argument("--cpu-sample", type=int, default=500_000, help="queries in the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extract", action="store_true", help="skip the configs[4] extraction inside the default run")
    ap.add_argument("--no-runs", action="store_true", help="skip the run-length workload inside the default run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0's share) to DIR/<name>.npy, at most 64 MB in all")
    return ap.parse_args()


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))


# ---- index image shared between the ranks of one box --------------------------------------------------

def get_image(sites, haplotypes, rank, world, barrier, model):
    """The Simple-SDS GBWT image. With several ranks only rank 0 needs it (it builds the index the others import, and
    runs the oracle); the others get None."""
    from synth import synth
    if rank != 0:
        return None, None
    t = time.time()
    img = synth.bubble_chain(sites, haplotypes, SEED, threads=(os.cpu_count() or 0) if world > 1 else 0, **model)
    log(f"[bench] generated index image: {img.nbytes / 1e9:.2f} GB in {time.time() - t:.1f} s")
    return img.array, img


# ---- clocks ---------------------------------------------------------------------------------------------

class ClockSampler:
    """Samples SM clock, power and throttle reasons through NVML every few milliseconds while the timed region
    runs (the same fields as the nvidia-smi line of B200_PROFILING.md, without the process start-up latency,
    so that even a 100 ms timed region gets samples)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, cuda_index):
        self.samples, self.handle, self.nv = [], None, None
        self._stop = threading.Event()
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(cuda_index).uuid)
            try:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(cuda_index)
            self.nv = pynvml
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        except Exception as exc:
            self.error = str(exc)
            self.handle = None

    def _run(self):
        nv, h = self.nv, self.handle
        while not self._stop.is_set():
            try:
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((time.time(), nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM),
                                     nv.nvmlDeviceGetPowerUsage(h) / 1000.0, mask))
            except Exception:
                pass
            time.sleep(0.004)

    def stop(self, t0, t1):
        if self.handle is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable: " + getattr(self, "error", "?")]}
        self._stop.set()
        self.thread.join(timeout=1.0)
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": float(self.sm_max), "reasons": ["no samples inside the timed region"]}
        reasons = set()
        for s in inside:
            for bit, name in self.REASONS.items():
                if s[3] & bit:
                    reasons.add(name)
        return {"sm_mhz": float(statistics.median(s[1] for s in inside)), "sm_max_mhz": float(self.sm_max),
                "power_w_max": max(s[2] for s in inside), "samples": len(inside), "reasons": sorted(reasons),
                "how": "NVML, 4 ms period, samples with timestamps inside the timed region only"}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


# ---- CPU side (oracle = C restatement of the reference path) ------------------------------------------

def cpu_find_baseline(image, sites, haplotypes, sample, steps=1, warmup=0, model=None):
    """Times the oracle (kind "port") on all host threads over `sample` queries per step."""
    from oracle import oracle as orc
    from synth import synth
    g = orc.GBWT.load(image, native=True)
    threads = orc.max_threads()
    pats = synth.patterns(sites, haplotypes, SEED, n=sample, k=K_LEN, seed_q=SEED_Q, q0=1 << 40, **(model or {}))
    for _ in range(warmup):
        g.find_extend_batch(pats, threads=threads)
    t = time.perf_counter()
    for _ in range(steps):
        out = g.find_extend_batch(pats, threads=threads)
    dt = time.perf_counter() - t
    assert np.all(out["end"] > out["start"])
    t1 = time.perf_counter()
    g.find_extend_batch(pats[: max(1, sample // 16)], threads=1)
    single = (time.perf_counter() - t1) / max(1, sample // 16)
    return {"value": sample * steps / dt, "unit": "queries/s", "cores": threads, "kind": "port",
            "sample": f"{sample} length-{K_LEN} patterns of the same workload per step, oracle/gbwt_oracle.c (-O3 -march=native, "
                      f"OpenMP dynamic over queries = rayon analogue), {threads} threads of {os.cpu_count()} host CPUs",
            "single_thread_us_per_query": single * 1e6, "single_thread_ns_per_node": single * 1e9 / K_LEN,
            "seconds": dt, "ms_per_step": dt / steps * 1e3}, g


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (C restatement; the Rust crate cannot be built here)."""
    if rank != 0:
        return
    sites, haplotypes, _ = resolve_workload(args)
    from synth import synth
    img = synth.bubble_chain(sites, haplotypes, SEED, **model_of(args))
    base, _ = cpu_find_baseline(img.array, sites, haplotypes, args.cpu_sample, steps=args.steps, warmup=args.warmup, model=model_of(args))
    line = {
        "impl": "reference", "metric": "gbwt_find_queries_per_s_k32", "value": base["value"], "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": dict(workload_config(args, sites, haplotypes, args.cpu_sample, "cpu"),
                       note=f"a rate: every step times a bounded sample of {args.cpu_sample} queries of the same workload (same index, same "
                            "pattern generator) against the GPU arm's 2^26 per GPU per step"),
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample", "single_thread_us_per_query",
                                              "single_thread_ns_per_node")},
        "e2e": {"value": base["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, arrays):
    """--dump-outputs: every device tensor of `arrays` as out_dir/<name>.npy in float64, which holds every value the timed
    paths return exactly. The inputs are the same from run to run, so two builds can be compared array by array. A tensor
    larger than its share of DUMP_BYTES is written as a fixed, seeded sample of its rows in ascending order, and the row
    numbers of the sample as <name>_rows.npy."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        n = t.shape[0]
        row_bytes = 8 * (t.numel() // n if n else 1)
        if n * row_bytes + 1024 <= share:
            host = t.cpu().numpy()
        else:
            rows = np.sort(np.random.default_rng(SEED).choice(n, size=(share - 2048) // (row_bytes + 8), replace=False))
            host = t[torch.from_numpy(rows).to(t.device)].cpu().numpy()
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, f"{name}.npy"), host.astype(np.float64))
    log(f"[bench] outputs of the last timed step written to {out_dir}: {', '.join(arrays)}")


def resolve_workload(args):
    sites, haplotypes, queries = WORKLOADS[args.workload]
    return args.sites or sites, args.haplotypes or haplotypes, args.queries or queries


def workload_config(args, sites, haplotypes, queries, where):
    model = model_of(args)
    if model["alt_ppm"]:
        what = (f"synthetic bubble-chain GBWT, {4 * sites + 1} node ids x {haplotypes} haplotypes ({sites} sites, alternative alleles of "
                f"frequency {model['alt_ppm'] / 1e6:g}, every {model['tri_mod']}th site tri-allelic, seed {SEED})")
    else:
        what = f"synthetic bubble-chain GBWT, {3 * sites + 1} nodes x {haplotypes} haplotypes ({sites} sites, iid alleles, seed {SEED})"
    return {"workload": what + f", length-{K_LEN} find/extend patterns sampled from the haplotypes (seed {SEED_Q})",
            "baseline_config": "BASELINE.json configs[3]" if args.workload == "find" else args.workload,
            "queries_per_gpu_per_step": queries, "pattern_len": K_LEN, "layout": args.layout, "where": where,
            "l2": "inputs larger than L2 (index + pattern batch >> 126 MB), no flush needed",
            "parallelism": f"index replicated, queries sharded over {args.gpus} GPU(s), no collective on the timed path"}


# ---- the GPU benchmark -------------------------------------------------------------------------------------

KERNEL_SOURCES = ("find_window.cu", "find_window.h", "find_lean.cuh", "record_scan.cuh", "layout.h", "kernels.cuh", "cabi.cu")


def kernel_source_hash():
    """sha256 over the sources the timed kernels are compiled from: ties a committed ncu capture to the code it measured."""
    import hashlib
    h = hashlib.sha256()
    for name in KERNEL_SOURCES:
        with open(os.path.join(ROOT, "gbwt-rs_b200", "csrc", name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def committed_traffic(kernel, queries, layout):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (profiles/find_window_traffic.json), scaled to
    this launch's query count -- or (None, why) when the capture was taken from other sources than the ones being timed."""
    try:
        with open(os.path.join(ROOT, "profiles", "find_window_traffic.json")) as f:
            prof = json.load(f)
    except Exception as exc:
        return None, f"no committed capture ({exc})"
    if prof.get("kernel") != kernel or prof.get("layout") != layout:
        return None, "the committed capture is of another kernel / layout"
    if prof.get("source_sha16") != kernel_source_hash():
        return None, "the committed capture was taken from other kernel sources than the ones being timed"
    per_query = (prof["dram_bytes_read"] + prof["dram_bytes_write"]) / prof["queries_per_launch"]
    return per_query * queries, f"ncu dram__bytes_read+write of one launch of {prof['queries_per_launch']} queries ({prof['captured']}), scaled by queries"


def main():
    args = parse_args()
    rank, world, local_rank = dist_env()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    import gbwt_rs_b200 as gb
    from synth import synth
    ncpu = os.cpu_count() or 8
    os.environ["GBWT_B200_BUILD_THREADS"] = str(ncpu)  # K0 runs on rank 0 only (the other ranks import its result)

    sites, haplotypes, Q = resolve_workload(args)

    def replicated_index(checkpoints, image_bytes=None):
        """The index on this rank's GPU: rank 0 parses the image, runs K0 and the checkpoint walk once, the other ranks
        import its arrays device to device (CUDA IPC + peer copies over NVLink) instead of repeating the host work."""
        barrier()  # (the first collective also sets up the NCCL communicator: keep that out of the build time)
        t = time.time()
        src = image if image_bytes is None else image_bytes
        if world == 1:
            return gb.GBWT.from_bytes(src, device=local_rank, layout=args.layout, checkpoints=checkpoints), time.time() - t
        box = [None]
        first = None
        if rank == 0:
            first = gb.GBWT.from_bytes(src, device=local_rank, layout=args.layout, checkpoints=checkpoints)
            log(f"[bench] rank 0 built the index in {time.time() - t:.1f} s; the other ranks copy it device to device")
            box[0] = first.export_ipc()
        dist.broadcast_object_list(box, src=0, device=dev)
        ix = first if rank == 0 else gb.GBWT.import_ipc(box[0], device=local_rank)
        barrier()  # rank 0 keeps its arrays alive until every rank has copied them
        return ix, max_over_ranks(time.time() - t)

    model = model_of(args)
    image, keep = get_image(sites, haplotypes, rank, world, barrier, model)
    index, build_s = replicated_index(True)
    stats = index.device_bytes()
    ckpt = index.checkpoint_info()
    if rank == 0:
        log(f"[bench] device index built in {build_s:.1f} s (checkpoint walk {ckpt['build_us'] / 1e6:.2f} s): {stats}")
    stream = torch.cuda.current_stream().cuda_stream

    if args.workload == "extract-dna":
        line = bench_extract_dna(args, index, image, sites, haplotypes, rank, world, local_rank, barrier, max_over_ranks, stats)
        if rank == 0:
            print(json.dumps(line), flush=True)
        return
    if args.workload == "extract":
        line = bench_extract(args, index, image, sites, haplotypes, rank, world, local_rank, barrier, max_over_ranks, stats)
        if rank == 0:
            print(json.dumps(line), flush=True)
        return

    # inputs resident in HBM before the timed region
    q0 = rank * Q
    d_pat = torch.empty((Q, K_LEN), dtype=torch.int64, device=dev)
    d_out = torch.empty((Q, 3), dtype=torch.int64, device=dev)
    synth.patterns_device(sites, haplotypes, SEED, Q, d_pat.data_ptr(), k=K_LEN, seed_q=SEED_Q, q0=q0, stream=stream, **model)
    torch.cuda.synchronize()

    def step():
        index.find_extend_device(d_pat.data_ptr(), Q, K_LEN, d_out.data_ptr(), stream)

    def timed_steps(fn, steps, warmup):
        """`steps` calls of fn bracketed by barrier + synchronize; returns (max-over-ranks total ms, per-step ms, clocks, launches)."""
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        sampler = ClockSampler(local_rank)
        time.sleep(0.25)
        launches0 = gb.kernel_launches()
        events = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        barrier(); torch.cuda.synchronize()
        t0 = time.time()
        events[0].record()
        for i in range(steps):
            fn()
            events[i + 1].record()
        torch.cuda.synchronize(); barrier()
        t1 = time.time()
        launches = gb.kernel_launches() - launches0
        clocks = sampler.stop(t0, t1)
        per_step = [events[i].elapsed_time(events[i + 1]) for i in range(steps)]
        return max_over_ranks(events[0].elapsed_time(events[-1])), per_step, clocks, launches

    total_ms, step_ms, clocks, launches = timed_steps(step, args.steps, args.warmup)
    value = Q * world * args.steps / (total_ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"states": d_out})  # (node, start, end) of every query

    # size-independent parity properties on the full batch (every sampled pattern occurs; state.node = last node)
    ok = bool(torch.all(d_out[:, 2] > d_out[:, 1]).item()) and bool(torch.equal(d_out[:, 0], d_pat[:, K_LEN - 1]))
    checksum = int((d_out[:, 2] - d_out[:, 1]).sum().item())
    if not ok:
        raise SystemExit("parity property violated: a sampled pattern was not found")
    want_out = d_out.clone()

    # the dominant kernel alone (CUDA events around its launch inside the library, GBWT_B200_WINDOW_STATS=1; these
    # three steps are outside the timed region because reading the counters synchronises the stream)
    os.environ["GBWT_B200_WINDOW_STATS"] = "1"
    w0 = index.window_info()
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    w1 = index.window_info()
    del os.environ["GBWT_B200_WINDOW_STATS"]
    win_launches = w1["launches"] - w0["launches"]
    kernel_ms = (w1["kernel_ns"] - w0["kernel_ns"]) / 1e6 / win_launches if win_launches else None
    deferred = (w1["deferred"] - w0["deferred"]) // 3 if win_launches else None

    # the same batch as 32-bit node identifiers (gbwt_b200_find_extend_u32_device): half the pattern bytes
    d_pat32 = d_pat.to(torch.int32)
    u32_ms, u32_steps, _, _ = timed_steps(lambda: index.find_extend_u32_device(d_pat32.data_ptr(), Q, K_LEN, d_out.data_ptr(), stream),
                                          max(3, min(args.steps, 10)), 2)
    if not torch.equal(d_out, want_out):
        raise SystemExit("32-bit pattern results differ from 64-bit pattern results")
    find_u32 = {"value": Q * world * len(u32_steps) / (u32_ms / 1e3), "unit": "queries/s", "ms_per_step": u32_ms / len(u32_steps),
                "api": "gbwt_b200_find_extend_u32_device"}

    # bidirectional searches on the same patterns (config 2's operation at config 4's size): bd_find of a random node of the
    # pattern, forward extensions to a random end, backward extensions to a random start, fused in one kernel
    bd = None
    if args.workload == "find":
        Qb = Q
        gen = torch.Generator(device=dev); gen.manual_seed(11 + rank)
        first = torch.randint(0, K_LEN, (Qb,), device=dev, generator=gen, dtype=torch.int64)
        start = (first.double() * torch.rand(Qb, device=dev, generator=gen, dtype=torch.float64)).long()
        end = first + 1 + ((K_LEN - 1 - first).double() * torch.rand(Qb, device=dev, generator=gen, dtype=torch.float64)).long()
        offs = torch.arange(Qb + 1, dtype=torch.int64, device=dev) * K_LEN
        d_bd = torch.empty((Qb, 6), dtype=torch.int64, device=dev)
        bd_ms, bd_steps, _, _ = timed_steps(lambda: index.bd_search_device(d_pat.data_ptr(), offs.data_ptr(), first.data_ptr(), start.data_ptr(),
                                                                           end.data_ptr(), Qb, d_bd.data_ptr(), stream), 3, 2)
        sizes_ok = bool(torch.all(d_bd[:, 2] > d_bd[:, 1]).item()) and bool(torch.equal(d_bd[:, 2] - d_bd[:, 1], d_bd[:, 5] - d_bd[:, 4]))
        if not sizes_ok:
            raise SystemExit("bidirectional search: a sampled subpath was not found, or forward and reverse ranges differ in size")
        bd_checked = 0
        if rank == 0:
            from oracle import oracle as orc
            nb = 20_000
            gb_oracle = orc.GBWT.load(image, native=True)
            want_bd = gb_oracle.bd_search_batch(d_pat[:nb].reshape(-1).cpu().numpy().view(np.uint64), (np.arange(nb + 1, dtype=np.uint64) * K_LEN),
                                                first[:nb].cpu().numpy().view(np.uint64), start[:nb].cpu().numpy().view(np.uint64),
                                                end[:nb].cpu().numpy().view(np.uint64))
            if not np.array_equal(d_bd[:nb].cpu().numpy().view(np.uint64).reshape(-1), want_bd.view(np.uint64).reshape(-1)):
                raise SystemExit("bidirectional search: parity failure against the oracle")
            bd_checked = nb
            del gb_oracle
        extensions = float((end - start - 1).sum().item())
        bd = {"value": Qb * world * len(bd_steps) / (bd_ms / 1e3), "unit": "searches/s", "ms_per_step": bd_ms / len(bd_steps),
              "searches_per_gpu_per_step": Qb, "lf_steps_per_s": extensions * world * len(bd_steps) / (bd_ms / 1e3),
              "api": "gbwt_b200_bd_search_device (bd_find + extend_forward* + extend_backward*, src/gbwt.rs:311-384)",
              "parity": f"every range non-empty and forward / reverse sizes equal on the full batch; first {bd_checked} searches bit-exact against the CPU oracle"}
        del first, start, end, offs, d_bd

    # end to end through the host C ABI with pinned buffers (H2D + kernels + D2H inside the timed region), both widths
    e2e = None
    if not args.no_e2e:
        e2e = bench_e2e(args, index, d_pat, want_out, Q, world, local_rank, barrier, max_over_ranks, sum_over_ranks)
    del d_pat32

    roofline, cpu = None, None
    if rank == 0:
        # algorithmic bytes per query of SURVEY.md 8(d), on the reference's compressed records, from a sample
        from oracle import oracle as orc
        t = time.time()
        sample_n = 1 << 18
        if args.no_cpu_baseline or world > 1:
            g = orc.GBWT.load(image, native=True)
        else:
            cpu, g = cpu_find_baseline(image, sites, haplotypes, args.cpu_sample, model=model)
        sample = synth.patterns(sites, haplotypes, SEED, n=sample_n, k=K_LEN, seed_q=SEED_Q, q0=q0, **model)
        bytes_per_query = g.find_extend_bytes(sample[:20_000]) / 20_000
        want = g.find_extend_batch(sample, threads=orc.max_threads())
        got = want_out[:sample_n].cpu().numpy().view(np.uint64)
        if not np.array_equal(got, want.view(np.uint64).reshape(-1, 3)):
            raise SystemExit("parity failure against the oracle on the sampled queries")
        peak, peak_src = measured_peak_gbs()
        kernel = "k_find_window" if win_launches else "k_find_extend"
        traffic, traffic_src = committed_traffic(kernel, Q, args.layout) if args.workload == "find" else (None, "not the headline workload")
        step_s = statistics.mean(step_ms) / 1e3
        launch_s = (kernel_ms / 1e3) if kernel_ms else step_s
        index_once = stats["descriptors"] + stats["bodies"] + stats["edges"] + stats.get("skips", 0)
        compulsory = Q * (K_LEN * 8 + 24) + index_once
        roofline = {"bound": "hbm", "kernel": kernel, "unit": "GB/s", "peak": peak, "peak_source": peak_src + " (of measured)",
                    # what the kernel really moves: measured DRAM bytes of one launch over its measured duration
                    "traffic": traffic, "traffic_source": traffic_src,
                    "achieved": (traffic / launch_s / 1e9) if traffic else None,
                    "frac": (traffic / launch_s / 1e9 / peak) if traffic else None,
                    # what it has to move at the very least: every pattern and result once, the index once
                    "compulsory_bytes": compulsory, "compulsory_frac": compulsory / step_s / 1e9 / peak,
                    "compulsory_frac_kernel_only": compulsory / launch_s / 1e9 / peak,
                    # SURVEY.md 8(d) accounting on the reference's compressed records (not a bound for this layout: the dense
                    # blocks answer a rank from 8 bytes and every record is read once per batch, so this is far above 1)
                    "algorithmic_bytes_per_query": bytes_per_query, "algorithmic_bytes_per_lf_step": bytes_per_query / K_LEN,
                    "algorithmic_x": bytes_per_query * Q / step_s / 1e9 / peak,
                    "launch_ms": launch_s * 1e3, "step_ms": step_s * 1e3, "launches_per_step": launches // max(1, args.steps),
                    "deferred_queries_per_step": deferred,
                    "note": "frac = measured DRAM bytes per launch (committed ncu capture of these kernel sources, hash-checked) / "
                            "live CUDA-event duration of the window kernel / measured HBM copy peak; compulsory_frac = (patterns + "
                            "results + index once) / whole step (sort + search) / peak: how far the step is from the bytes it cannot avoid"}
        log(f"[bench] oracle sample + cpu baseline took {time.time() - t:.1f} s")

    # BASELINE.json configs[4] in the same run: extraction of all forward haplotype paths, partitioned by path
    extract = None
    if args.workload == "find" and not args.no_extract:
        del d_pat, d_out, want_out
        torch.cuda.empty_cache()
        extract = bench_extract_inline(args, index, image, sites, haplotypes, rank, world, local_rank, barrier, max_over_ranks, ckpt, stats,
                                       replicated_index)

    # the run-length workload in the same run (low-frequency alleles, tri-allelic sites: records the dense bitvector does not cover)
    find_runs = None
    if args.workload == "find" and not args.no_runs:
        del index
        torch.cuda.empty_cache()
        find_runs = bench_find_runs(args, rank, world, local_rank, barrier, max_over_ranks, replicated_index)

    if rank == 0:
        line = {
            "metric": "gbwt_find_queries_per_s_k32", "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": workload_config(args, sites, haplotypes, Q, "inputs and outputs resident in HBM"),
            "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
            "extra": {"lf_steps_per_s": value * K_LEN, "find_u32": find_u32, "bd_search": bd, "extract": extract, "find_runs": find_runs,
                      "occurrences_checksum": checksum, "index_device_bytes": stats, "index_build_s": build_s,
                      "checkpoints": ckpt, "window": {k: w1[k] for k in ("window_records", "margin", "threads", "smem_bytes", "windows")},
                      "step_ms": step_ms, "arithmetic": "u64 node identifiers and offsets at the ABI, 32-bit inside the kernels "
                                                        "(an index that does not fit is rejected at load)",
                      "parity": f"all patterns found, state.node == last node on the full batch; first {1 << 18} queries bit-exact "
                                "against the CPU oracle; 32-bit and host-path results identical to the device-path results"},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def bench_e2e(args, index, d_pat, want_out, Q, world, local_rank, barrier, max_over_ranks, sum_over_ranks):
    """The same metric through the host entry points (pinned host buffers in, pinned host buffers out): the 32-bit call
    is the headline (what a caller that narrows its node identifiers once pays), the 64-bit call beside it, and the
    plain H2D copy rate of the same buffer, which is the bound for both."""
    import torch
    import gbwt_rs_b200 as gb
    lib = gb.library()
    Qe = min(args.e2e_queries, Q)
    e2e_steps = max(3, min(args.steps, 10))
    out = {}
    for width in ("u32", "u64"):
        dtype = torch.int32 if width == "u32" else torch.int64
        h_pat = torch.empty((Qe, K_LEN), dtype=dtype).pin_memory()
        h_out = torch.empty((Qe, 3), dtype=torch.int64).pin_memory()
        h_pat.copy_(d_pat[:Qe].to(dtype))
        fn = lib.gbwt_b200_find_extend_u32 if width == "u32" else lib.gbwt_b200_find_extend

        def e2e_step():
            rc = fn(index._h, h_pat.data_ptr(), Qe, K_LEN, h_out.data_ptr())
            if rc != 0:
                raise SystemExit(f"gbwt_b200_find_extend failed: {lib.gbwt_b200_last_error().decode()}")
        e2e_step()
        barrier(); torch.cuda.synchronize()
        te = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - te)
        barrier()
        if not torch.equal(h_out, want_out[:Qe].cpu()):
            raise SystemExit("host-path results differ from device-path results")
        # the wire: the same pinned buffer copied to the device and nothing else, all ranks at once
        d_tmp = torch.empty_like(h_pat, device=d_pat.device)
        d_tmp.copy_(h_pat, non_blocking=True)
        barrier(); torch.cuda.synchronize()
        tw = time.perf_counter()
        for _ in range(3):
            d_tmp.copy_(h_pat, non_blocking=True)
        torch.cuda.synchronize()
        wire_s = max_over_ranks(time.perf_counter() - tw) / 3
        barrier()
        item = K_LEN * (4 if width == "u32" else 8)
        out[width] = {"value": Qe * world * e2e_steps / dt, "unit": "queries/s", "h2d_bytes_per_step": Qe * item,
                      "d2h_bytes_per_step": Qe * 24, "h2d_wire_gbs_per_gpu": Qe * item / wire_s / 1e9,
                      "wire_bound_queries_per_s": Qe * world / wire_s,
                      "api": f"gbwt_b200_find_extend{'_u32' if width == 'u32' else ''} (host pointers, pinned), chunked H2D/kernels/D2H on alternating streams"}
        del h_pat, h_out, d_tmp
    e2e = dict(out["u32"])
    e2e.update({"queries_per_gpu_per_step": Qe, "steps": e2e_steps, "u64": out["u64"],
                "limiter": "host-to-device copy of the patterns (PCIe): compare value with wire_bound_queries_per_s, the rate at which "
                           "the same pinned buffer is copied with nothing else running"})
    return e2e


def bench_find_runs(args, rank, world, local_rank, barrier, max_over_ranks, replicated_index):
    """The same metric on the run-length workload (WORKLOADS["find-runs"]): alternative alleles of frequency 0.05 and every
    tenth site tri-allelic, so that the anchors are not all plain bitvectors -- three-edge records (DENSE4), byte-per-run
    bodies and their checkpoint tables are on the path. Device-resident patterns, weak scaling like the headline."""
    import torch
    import gbwt_rs_b200 as gb
    from synth import synth
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.current_stream().cuda_stream
    sites, haplotypes, Q = WORKLOADS["find-runs"]
    model = MODELS["find-runs"]
    Q = min(Q, args.queries) if args.queries else Q
    img = None
    if rank == 0:
        img = synth.bubble_chain(sites, haplotypes, SEED, threads=(os.cpu_count() or 0) if world > 1 else 0, **model)
    index, build_s = replicated_index(False, img.array if img is not None else None)
    stats = index.device_bytes()
    d_pat = torch.empty((Q, K_LEN), dtype=torch.int64, device=dev)
    d_out = torch.empty((Q, 3), dtype=torch.int64, device=dev)
    synth.patterns_device(sites, haplotypes, SEED, Q, d_pat.data_ptr(), k=K_LEN, seed_q=SEED_Q, q0=rank * Q, stream=stream, **model)
    torch.cuda.synchronize()
    steps = max(3, min(args.steps, 5))
    for _ in range(2):
        index.find_extend_device(d_pat.data_ptr(), Q, K_LEN, d_out.data_ptr(), stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(); torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        index.find_extend_device(d_pat.data_ptr(), Q, K_LEN, d_out.data_ptr(), stream)
    e1.record()
    torch.cuda.synchronize(); barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    if not (bool(torch.all(d_out[:, 2] > d_out[:, 1]).item()) and bool(torch.equal(d_out[:, 0], d_pat[:, K_LEN - 1]))):
        raise SystemExit("run-length workload: a sampled pattern was not found")
    os.environ["GBWT_B200_WINDOW_STATS"] = "1"
    w0 = index.window_info()
    index.find_extend_device(d_pat.data_ptr(), Q, K_LEN, d_out.data_ptr(), stream)
    torch.cuda.synchronize()
    w1 = index.window_info()
    del os.environ["GBWT_B200_WINDOW_STATS"]
    checked = 0
    if rank == 0:
        from oracle import oracle as orc
        g = orc.GBWT.load(img.array, native=True)
        sample_n = 1 << 18
        sample = synth.patterns(sites, haplotypes, SEED, n=sample_n, k=K_LEN, seed_q=SEED_Q, q0=0, **model)
        want = g.find_extend_batch(sample, threads=orc.max_threads())
        if not np.array_equal(d_out[:sample_n].cpu().numpy().view(np.uint64), want.view(np.uint64).reshape(-1, 3)):
            raise SystemExit("run-length workload: parity failure against the oracle")
        checked = sample_n
    res = {"metric": "gbwt_find_queries_per_s_k32", "value": Q * world / (ms / 1e3), "unit": "queries/s", "ms_per_step": ms, "steps": steps,
           "queries_per_gpu_per_step": Q,
           "workload": f"{4 * sites + 1} node ids x {haplotypes} haplotypes, alternative alleles of frequency {model['alt_ppm'] / 1e6:g}, every "
                       f"{model['tri_mod']}th site tri-allelic; length-{K_LEN} patterns sampled from the haplotypes",
           "index_device_bytes": stats, "index_build_s": build_s,
           "window_kernel_ms": (w1["kernel_ns"] - w0["kernel_ns"]) / 1e6 if w1["launches"] > w0["launches"] else None,
           "deferred_queries_per_step": w1["deferred"] - w0["deferred"],
           "parity": f"all patterns found, state.node == last node on the full batch; first {checked} queries bit-exact against the CPU oracle"}
    del d_pat, d_out, index
    torch.cuda.empty_cache()
    return res


def bench_extract_inline(args, index, image, sites, haplotypes, rank, world, local_rank, barrier, max_over_ranks, ckpt, stats,
                         replicated_index):
    """configs[4] inside the default run: every forward haplotype path, partitioned by path over the ranks (strong scaling).
    warm = the index as the library builds it (path checkpoints from the load-time walk: sequences are extracted as
    independent segments); cold = a fresh handle WITHOUT checkpoints and without remembered lengths (one dependent chain per
    path), first call and second call."""
    import torch
    import gbwt_rs_b200 as gb
    from synth import synth
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.current_stream().cuda_stream
    lo, hi = gb.shard_range(haplotypes, rank, world)
    m = hi - lo
    length = 2 * sites + 1
    ids = (torch.arange(lo, hi, dtype=torch.int64, device=dev) * 2)
    offs = torch.arange(m + 1, dtype=torch.int64, device=dev) * length
    nodes = torch.empty(m * length, dtype=torch.int64, device=dev)
    lens = torch.empty(m, dtype=torch.int64, device=dev)

    def run(ix, steps, warmup):
        for _ in range(warmup):
            ix.extract_device(ids.data_ptr(), m, offs.data_ptr(), nodes.data_ptr(), lens.data_ptr(), stream)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            ix.extract_device(ids.data_ptr(), m, offs.data_ptr(), nodes.data_ptr(), lens.data_ptr(), stream)
        e1.record()
        torch.cuda.synchronize(); barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps

    steps = max(3, min(args.steps, 10))
    nodes.zero_()
    warm_ms = run(index, steps, 2)
    if not bool(torch.all(lens == length).item()):
        raise SystemExit("extraction: wrong sequence lengths")
    # parity: 8 whole paths of this rank against the oracle (rank 0 checks its own; every rank checks the generator)
    picks = sorted(set(int(x) for x in np.linspace(0, m - 1, 8)))
    for j in picks[:2]:
        got = nodes[j * length:(j + 1) * length].cpu().numpy().view(np.uint64)
        if not np.array_equal(got, synth.sequence(sites, haplotypes, SEED, 2 * (lo + j))):
            raise SystemExit("extraction: a path differs from the generator's haplotype")
    oracle_paths = 0
    if rank == 0:
        from oracle import oracle as orc
        g = orc.GBWT.load(image, native=True)
        want_ids = np.array([2 * (lo + j) for j in picks], dtype=np.uint64)
        w_off, w_nodes = g.extract_batch(want_ids, threads=len(picks))
        for t, j in enumerate(picks):
            got = nodes[j * length:(j + 1) * length].cpu().numpy().view(np.uint64)
            if not np.array_equal(got, w_nodes[int(w_off[t]):int(w_off[t + 1])]):
                raise SystemExit("extraction: a path differs from the oracle's")
        oracle_paths = len(picks)
    warm_sum = int(nodes.sum().item())
    # cold: a fresh handle without checkpoints
    cold, cold_build_s = replicated_index(False)
    nodes.zero_()
    cold_first_ms = run(cold, 1, 0)
    if int(nodes.sum().item()) != warm_sum:
        raise SystemExit("extraction: chain walks and checkpointed extraction disagree")
    cold_second_ms = run(cold, 1, 0)
    if int(nodes.sum().item()) != warm_sum:
        raise SystemExit("extraction: two-ended walks and checkpointed extraction disagree")
    del cold
    total_nodes = haplotypes * length
    peak, _ = measured_peak_gbs()
    sm_mhz = 1965.0
    # latency rooflines (dependent-load latencies measured with tools/microbench on this pool's B200: L2 291, HBM 813 cycles)
    lat_l2, lat_hbm = 291.0, 813.0
    props = torch.cuda.get_device_properties(local_rank)

    def latency_bound(chains, nodes_per_trip, latency_cycles):
        return chains * nodes_per_trip / (latency_cycles / (sm_mhz * 1e6)) * world

    cold_chains = m                                   # one warp-wide chain per path, two nodes per dependent load (two-hop shortcuts)
    # lanes resident: 1024 per SM in the window kernel (256 or more paths per GPU), 5 CTAs of 256 in the one-lane kernel
    warm_chains = min(m * max(1, ckpt["max_segments"]), props.multi_processor_count * (1024 if m >= 96 else 1280))
    out_bytes = total_nodes * 8 + (stats["descriptors"] + stats["bodies"] + stats.get("skips", 0)) // 2 * world
    res = {
        "metric": "gbwt_extract_lf_steps_per_s", "unit": "LF steps/s", "scaling": "strong", "paths_per_gpu": m, "nodes_per_path": length,
        "warm_lf_steps_per_s": total_nodes / (warm_ms / 1e3), "warm_ms": warm_ms,
        "warm_kernel": "k_extract_window" if m >= 96 else "k_extract_checkpointed",
        "cold_lf_steps_per_s": total_nodes / (cold_first_ms / 1e3), "cold_first_call_ms": cold_first_ms,
        "cold_second_call_lf_steps_per_s": total_nodes / (cold_second_ms / 1e3), "cold_second_call_ms": cold_second_ms,
        "checkpoint_build_s": ckpt["build_us"] / 1e6, "checkpoint_interval": ckpt["interval"], "checkpoint_bytes": ckpt["bytes"],
        "cold_index_build_s": cold_build_s,
        "frac_bytes": out_bytes / (warm_ms / 1e3) / 1e9 / (peak * world),
        # (latency rooflines of the one-lane kernel only: a step of the window kernel is a shared-memory round trip, its bounds
        # are the bytes it writes and its issue slots)
        "frac_latency_hbm": total_nodes / (warm_ms / 1e3) / latency_bound(warm_chains, 1.0, lat_hbm) if m < 96 else None,
        "frac_latency_l2": total_nodes / (warm_ms / 1e3) / latency_bound(warm_chains, 1.0, lat_l2) if m < 96 else None,
        "cold_frac_latency_hbm": total_nodes / (cold_first_ms / 1e3) / latency_bound(cold_chains, 2.0, lat_hbm),
        "cold_frac_latency_l2": total_nodes / (cold_first_ms / 1e3) / latency_bound(cold_chains, 2.0, lat_l2),
        "oracle_checked_paths": oracle_paths,
        "note": "warm: every sequence cut into independent segments at the checkpoints the index was built with (build time above; "
                "the checkpoints are part of the immutable index, not a cache). With 96 or more paths per GPU a CTA takes one "
                "segment of up to 512 sequences, stages the records they walk in shared memory and the lanes step from there "
                "(k_extract_window); with fewer, one lane per segment walks from global memory (k_extract_checkpointed: two "
                "dependent loads per two-node step, latency bound = 1 node per round trip x lanes in flight). cold: a handle created "
                "without checkpoints, one dependent chain per path (two-hop steps). A path is only walked from both ends once BOTH "
                "of its strands have been walked whole and their signatures agree; this run extracts the forward strands only, so "
                "the second cold call repeats the first. frac_bytes = (8-byte nodes written + forward half of the index read once) "
                "/ time / measured HBM peak. Cold and warm produce identical bytes (checked); 8 whole paths compared with the CPU "
                "oracle on rank 0",
    }
    del nodes
    torch.cuda.empty_cache()
    return res


def bench_extract(args, index, image, sites, haplotypes, rank, world, local_rank, barrier, max_over_ranks, stats):
    """configs[4]: extraction of all forward haplotype paths via LF, partitioned by path."""
    import torch
    import gbwt_rs_b200 as gb
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.current_stream().cuda_stream
    lo, hi = gb.shard_range(haplotypes, rank, world)
    m = hi - lo
    length = 2 * sites + 1
    ids = (torch.arange(lo, hi, dtype=torch.int64, device=dev) * 2)
    offs = torch.arange(m + 1, dtype=torch.int64, device=dev) * length
    nodes = torch.empty(m * length, dtype=torch.int64, device=dev)
    lens = torch.empty(m, dtype=torch.int64, device=dev)

    def step():
        index.extract_device(ids.data_ptr(), m, offs.data_ptr(), nodes.data_ptr(), lens.data_ptr(), stream)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    launches0 = gb.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(); torch.cuda.synchronize()
    t0 = time.time()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize(); barrier()
    t1 = time.time()
    total_ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop(t0, t1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"nodes": nodes, "lengths": lens})
    assert bool(torch.all(lens == length).item())
    from synth import synth
    first = nodes[:length].cpu().numpy().view(np.uint64)
    assert np.array_equal(first, synth.sequence(sites, haplotypes, SEED, 2 * lo))
    steps_total = haplotypes * length * args.steps
    value = steps_total / (total_ms / 1e3)
    roofline = None
    if rank == 0:
        from oracle import oracle as orc
        g = orc.GBWT.load(image, native=True)
        sample_ids = np.arange(0, 2 * haplotypes, max(2, 2 * (haplotypes // 8)), dtype=np.uint64)
        per_step = g.extract_bytes(sample_ids) / (len(sample_ids) * length)
        peak, src = measured_peak_gbs()
        achieved = per_step * haplotypes * length / world / (total_ms / args.steps / 1e3) / 1e9
        kernel = ("k_extract_window" if m >= 96 else "k_extract_checkpointed") if index.checkpoint_info()["present"] else "k_extract"
        written = haplotypes * length * 8 / world / (total_ms / args.steps / 1e3) / 1e9
        roofline = {"bound": "hbm", "kernel": kernel, "achieved": written, "peak": peak, "unit": "GB/s", "frac": written / peak,
                    "traffic": None, "peak_source": src, "algorithmic_bytes_per_lf_step": per_step, "algorithmic_x": achieved / peak,
                    "note": "achieved = 8-byte nodes written / time (what the checkpointed kernels are bound by); algorithmic_x = SURVEY.md "
                            "8(d)'s bytes on the reference's compressed records / time / peak. A walk without checkpoints is a dependent "
                            "chain: its bound is chains in flight / access latency (extra.extract of the default run)"}
    return {"metric": "gbwt_extract_lf_steps_per_s", "value": value, "unit": "LF steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"extraction of all {haplotypes} forward haplotype paths ({length} nodes each) of the "
                                   f"{3 * sites + 1}-node bubble-chain GBWT", "baseline_config": "BASELINE.json configs[4]",
                       "paths_per_gpu": m, "layout": args.layout,
                       "note": "the index carries path checkpoints (built at load): every sequence is extracted as independent segments"},
            "gpu_launches": gb.kernel_launches() - launches0, "roofline": roofline, "clocks": clocks,
            "extra": {"index_device_bytes": stats}}


def bench_extract_dna(args, index, image, sites, haplotypes, rank, world, local_rank, barrier, max_over_ranks, stats):
    """SURVEY.md 8(f) next-3: DNA-level extraction (extract_sequence of src/bin/gbz-extract.rs:173-189) of all forward
    haplotype paths of the configs[4] graph with synthetic node labels, partitioned by path."""
    import torch
    import gbwt_rs_b200 as gb
    from synth import synth
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.current_stream().cuda_stream
    starts, labels = synth.node_labels(3 * sites + 1, seed=SEED, max_anchor=32)
    index.attach_graph(starts, labels)
    lo, hi = gb.shard_range(haplotypes, rank, world)
    m = hi - lo
    length = 2 * sites + 1
    ids = (torch.arange(lo, hi, dtype=torch.int64, device=dev) * 2)
    lens = torch.empty(m, dtype=torch.int64, device=dev)
    index.dna_lengths_device(ids.data_ptr(), m, lens.data_ptr(), stream)
    torch.cuda.synchronize()
    offs = torch.zeros(m + 1, dtype=torch.int64, device=dev)
    offs[1:] = torch.cumsum(lens, 0)
    total_bytes = int(offs[-1].item())
    out = torch.empty(total_bytes, dtype=torch.uint8, device=dev)
    got = torch.empty(m, dtype=torch.int64, device=dev)

    def step():
        index.extract_dna_device(ids.data_ptr(), m, 0, offs.data_ptr(), out.data_ptr(), got.data_ptr(), stream)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    launches0 = gb.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(); torch.cuda.synchronize()
    t0 = time.time()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize(); barrier()
    t1 = time.time()
    total_ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop(t0, t1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"dna": out, "lengths": got})
    assert bool(torch.all(got == lens).item())
    launches = gb.kernel_launches() - launches0
    # the same walks without the byte copy (label ranges and lengths only, one-ended), for the cost split
    l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0.record()
    index.dna_lengths_device(ids.data_ptr(), m, got.data_ptr(), stream)
    l1.record()
    torch.cuda.synchronize()
    lengths_only_ms = l0.elapsed_time(l1)
    all_bytes = max_over_ranks(float(total_bytes)) * world if world > 1 else float(total_bytes)
    value = all_bytes * args.steps / (total_ms / 1e3)
    cpu_baseline = None
    if rank == 0:
        # parity of the first and last path of this rank against the oracle, and the CPU baseline on a sample
        from oracle import oracle as orc
        gbz = synth.gbz_image(image, starts, labels, 3, as_image=True)
        g = orc.GBWT.load(gbz.array, native=True)
        sample = np.array([2 * lo, 2 * (hi - 1)], dtype=np.uint64)
        t = time.time()
        w_offsets, w_bytes, _ = g.extract_dna_batch(sample, 0, threads=2)
        dt = time.time() - t
        for j, i in enumerate((0, m - 1)):
            a, b = int(offs[i].item()), int(offs[i + 1].item())
            assert np.array_equal(out[a:b].cpu().numpy(), w_bytes[int(w_offsets[j]):int(w_offsets[j + 1])])
        cpu_baseline = {"value": float(w_offsets[-1]) / dt, "unit": "bases/s", "cores": 2, "kind": "port",
                        "sample": "2 of the paths, one thread each"}
    return {"metric": "gbz_extract_dna_bases_per_s", "value": value, "unit": "bases/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"DNA sequences of all {haplotypes} forward haplotype paths ({length} nodes, "
                                   f"{total_bytes // max(1, m)} bases each) of the {3 * sites + 1}-node bubble-chain GBZ",
                       "paths_per_gpu": m, "layout": args.layout, "label_bytes": int(starts[-1]),
                       "kernel": "k_extract_dna_checkpointed" if index.checkpoint_info()["present"] else "k_extract_dna_relay",
                       "note": "with path checkpoints (the default for an index of this size) the DNA position of every checkpoint is counted "
                               "when the labels are attached and every segment is spelled independently (k_extract_dna_checkpointed); "
                               "without them sequence and DNA lengths are known from the dna_lengths call that sized the output and every "
                               "path is walked from both ends by two warps that relay their nodes to a spelling warp (k_extract_dna_relay)"},
            "gpu_launches": launches, "clocks": clocks, "cpu_baseline": cpu_baseline,
            "extra": {"lf_steps_per_s": haplotypes * length * args.steps / (total_ms / 1e3), "lengths_only_ms": lengths_only_ms,
                      "index_device_bytes": stats,
                      "output_bytes_per_gpu": total_bytes}}


if __name__ == "__main__":
    main()
