#!/usr/bin/env python
"""bench.py -- headline benchmark of sourmash_b200 (contract: see the task statement / DESIGN.md §Measurement).

Primary workload (BASELINE.json configs[2]): `compare` of 10 000 synthetic FracMinHash sketches
(k=31, scaled=1000, ~5000 hashes each, 100 families) -> all-vs-all Jaccard matrix; metric
sketch-pairs/s.  Secondary workload (configs[1], reported under "sketch"): `sketch dna`
k=21,31,51 scaled=1000 over 100 synthetic 5 Mbp genomes; metric k-mers hashed/s.

    python bench.py --gpus 1 --steps 5 --warmup 3                  # this framework on cuda:0
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                           # CPU restatement on host cores

One JSON line on stdout (rank 0).  Only the cpu_baseline / --impl reference legs touch oracle/.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SKETCHES = 10_000
KSIZES = (21, 31, 51)
N_GENOMES = 100
COMPARE_WORKLOAD = ("configs[2]: compare 10000 synthetic sketches (k=31, scaled=1000, ~5000 hashes, "
                    "100 families) all-vs-all jaccard float64 matrix")
SKETCH_WORKLOAD = "configs[1]: sketch dna k=21,31,51 scaled=1000 on 100 synthetic 5 Mbp genomes"
N_DB_SEARCH, N_DB_GATHER, N_QUERY_SEARCH = 300_000, 50_000, 10_000_000   # configs[3] / configs[4] shapes
SM_COUNT = 148                                        # B200
GENOME_LEN = 5_000_000
SCALED = 1000


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------- --dump-outputs
DUMP_LIMIT_BYTES = 64 << 20
DUMP_SEED = 0
_OUTPUTS = {}


def keep_output(name, array):
    "an array the timed path returned in its last step, saved as <name>.npy by write_outputs()"
    array = np.ascontiguousarray(array)
    assert array.dtype in (np.float32, np.float64), (name, array.dtype)
    _OUTPUTS[name] = array


def u64_as_float64(name, values):
    "uint64 values as two exact float64 arrays (<name>_hi32, <name>_lo32): float64 holds 53 bits, a hash has 64"
    values = np.asarray(values, dtype=np.uint64)
    keep_output(name + "_hi32", (values >> np.uint64(32)).astype(np.float64))
    keep_output(name + "_lo32", (values & np.uint64(0xFFFFFFFF)).astype(np.float64))


def write_outputs(directory):
    total = sum(a.nbytes for a in _OUTPUTS.values())
    assert total <= DUMP_LIMIT_BYTES, "outputs to dump: %d bytes, more than %d" % (total, DUMP_LIMIT_BYTES)
    os.makedirs(directory, exist_ok=True)
    for name, array in sorted(_OUTPUTS.items()):
        np.save(os.path.join(directory, name + ".npy"), array)
    log(f"[bench] wrote {len(_OUTPUTS)} output arrays ({total} bytes) to {directory}")


# stdout carries exactly one JSON line: keep a private handle to the real stdout and point fd 1
# at stderr, so that library banners (e.g. "NCCL version ..." printed from C) cannot pollute it.
_JSON_FD = None


def protect_stdout():
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit_json(obj):
    data = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """`nvidia-smi -lms 20` running for the whole benchmark (it needs ~0.3 s to deliver its first
    line, longer than some timed regions); every timed region reports the samples whose arrival
    time falls inside it, widened to the nearest samples when the region is shorter than the
    sampling period."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def window(self, t_begin, t_end):
        "Clock statistics of the samples taken in [t_begin, t_end] (monotonic seconds)."
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)                                  # let the last in-region line arrive
        rows = list(self.rows)
        inside = [r for r in rows if t_begin <= r[0] <= t_end + 0.03]
        note = "timed region"
        if len(inside) < 2:                               # region shorter than two sampling periods
            mid = 0.5 * (t_begin + t_end)
            inside = sorted(rows, key=lambda r: abs(r[0] - mid))[:3]
            note = "3 samples nearest to the timed region (region shorter than two 20 ms sampling periods)"
        sm, mx, reasons = [], None, set()
        for _, r in inside:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, v in zip(self.NAMES, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "samples": len(sm), "reasons": sorted(reasons), "window": note}


# ----------------------------------------------------------------------------- workloads
def compare_workload():
    from sourmash_b200.synth import synth_sketches
    t = time.time()
    h, off = synth_sketches(N_SKETCHES)
    log(f"[bench] compare workload: {N_SKETCHES} sketches, {len(h)} hashes ({time.time() - t:.1f}s)")
    return h, off


def sketch_workload(n_genomes=N_GENOMES):
    from sourmash_b200.synth import synth_genome
    t = time.time()
    total = n_genomes * GENOME_LEN
    seqs = np.empty(total, dtype=np.uint8)
    for g in range(n_genomes):
        seqs[g * GENOME_LEN:(g + 1) * GENOME_LEN] = synth_genome(GENOME_LEN, 1000 + g)
    offs = (np.arange(n_genomes + 1, dtype=np.uint64) * np.uint64(GENOME_LEN))
    log(f"[bench] sketch workload: {n_genomes} genomes x {GENOME_LEN} bp ({time.time() - t:.1f}s)")
    return seqs, offs


def host_cores():
    """Usable host threads: the smallest of cpu_count, the affinity mask (the one the process started with) and the
    cgroup CPU quota."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(_ALL_CPUS if _ALL_CPUS is not None else os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        pass
    return n


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def git_blob_hash(path):
    "the id `git hash-object` gives the file: sha1 over 'blob <size>\\0' + content"
    import hashlib
    with open(path, "rb") as fh:
        data = fh.read()
    return hashlib.sha1(b"blob %d\0" % len(data) + data).hexdigest()


def ncu_record(key):
    """An ncu-measured constant (DRAM bytes per launch, warp instructions per k-mer) from profiles/ncu_traffic.json,
    or None when it is absent or STALE: every entry lists the kernel source files it was measured on with their
    git blob ids, and counts only while those files are byte-identical (scripts/record_traffic.py writes entries)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as fh:
        entry = json.load(fh).get("entries", {}).get(key)
    if not entry or not entry.get("files"):
        return None
    for rel, blob in entry["files"].items():
        path = os.path.join(ROOT, rel)
        if not os.path.exists(path) or git_blob_hash(path) != blob:
            return None
    return entry


def ncu_traffic(key):
    entry = ncu_record(key)
    return entry["value"] if entry else None


def ncu_source(key):
    entry = ncu_record(key)
    return entry.get("source") if entry else None


# ----------------------------------------------------------------------------- reference arm
def cpu_compare_sample(h, off, ncores, target_pairs):
    """Time the oracle's compare_serial restatement on rows [0, R) (all columns j > i)."""
    import oracle as orc
    all_host_cpus()
    n = len(off) - 1
    rows, pairs = 0, 0
    while rows < n and pairs < target_pairs:
        pairs += n - 1 - rows
        rows += 1
    t = time.perf_counter()
    want = orc.compare_all_pairs(h, off, first_row=0, n_rows=rows, nthreads=ncores)
    dt = time.perf_counter() - t
    return pairs, dt, f"rows 0..{rows - 1} x all later columns of the {n}-sketch matrix = {pairs} pairs", want[:rows]


def cpu_sketch_sample(seqs, offs, ncores, n_genomes):
    import oracle as orc
    all_host_cpus()
    sub_off = offs[: n_genomes + 1]
    sub = seqs[: int(sub_off[-1])]
    mx = orc.max_hash_for_scaled(SCALED)
    kmers, t, sketches = 0, time.perf_counter(), {}
    for k in KSIZES:
        sketches[k] = orc.sketch_batch(sub, sub_off, k, mx, nthreads=ncores, cap_per_seq=20000)
        kmers += int(sum(int(sub_off[i + 1] - sub_off[i]) - k + 1 for i in range(n_genomes)))
    dt = time.perf_counter() - t
    return kmers, dt, f"{n_genomes} of the {N_GENOMES} genomes x k={list(KSIZES)} = {kmers} k-mers", sketches


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncores = host_cores()
    if args.workload == "compare":
        h, off = compare_workload()
        target = int(1.5e5 * ncores)            # ~8 s per step at ~1.5e4 pairs/s/core
        times = []
        for i in range(args.warmup + args.steps):
            units, dt, sample, _rows = cpu_compare_sample(h, off, ncores, target)
            if i >= args.warmup:
                times.append(dt)
        metric, unit = "sketch-pairs/sec (compare)", "pairs/s"
        config = {"workload": COMPARE_WORKLOAD, "n_sketches": N_SKETCHES,
                  "pairs_per_step": N_SKETCHES * (N_SKETCHES - 1) // 2,
                  "parallelism": "%d host threads (OpenMP over rows)" % ncores}
    else:
        ng = N_GENOMES                           # the whole configs[1] workload (a few seconds on 16 cores)
        seqs, offs = sketch_workload(ng)
        times = []
        for i in range(args.warmup + args.steps):
            units, dt, sample, _sk = cpu_sketch_sample(seqs, offs, ncores, ng)
            if i >= args.warmup:
                times.append(dt)
        metric, unit = "k-mers hashed/sec (sketch)", "k-mers/s"
        config = {"workload": SKETCH_WORKLOAD, "parallelism": "%d host threads (one genome per thread)" % ncores}
    ms = 1000.0 * float(np.mean(times))
    value = units / (ms / 1000.0)
    line = {"impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": value, "unit": unit, "cores": ncores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "CPU restatement of src/core (oracle/oracle.c, OpenMP), not the Rust binary: no Rust toolchain in the image"}
    emit_json(line)


_ALL_CPUS = None


def all_host_cpus():
    "give the process back every CPU it started with (the CPU arm uses all host threads it can)"
    if _ALL_CPUS is not None:
        try:
            os.sched_setaffinity(0, _ALL_CPUS)
        except OSError:
            pass


def bind_to_gpu_cpus(torch, local_rank):
    """Pin this process to the CPUs next to its GPU (what `numactl` does for a PCIe-bound job): the pinned host buffers
    of the end-to-end legs are then allocated on the GPU's own NUMA node.  Best effort: returns a short description."""
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(local_rank).uuid)
        handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        global _ALL_CPUS
        _ALL_CPUS = os.sched_getaffinity(0)
        before = len(_ALL_CPUS)
        pynvml.nvmlDeviceSetCpuAffinity(handle)
        return "cpu affinity %d -> %d cpus (GPU-local)" % (before, len(os.sched_getaffinity(0)))
    except Exception as exc:                                       # noqa: BLE001
        return "cpu affinity unchanged (%s)" % type(exc).__name__


# ----------------------------------------------------------------------------- B200 arm
def run_b200(args):
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    log("[bench] rank %d: %s" % (rank, bind_to_gpu_cpus(torch, local_rank)))
    dist = None
    if world > 1:
        # keep stdout clean for the single JSON line: NCCL's banner / debug output goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from sourmash_b200 import batch as B
    B.set_device(local_rank)
    stream = torch.cuda.current_stream()
    B.set_stream(stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                                   # runs until the process exits (daemon reader)
        import atexit
        atexit.register(sampler.stop)

    def timed(step_fn, steps, warmup):
        for _ in range(warmup):
            step_fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = B.kernel_launches()
        t_begin = time.monotonic()
        e0.record(stream)
        extra = [step_fn() for _ in range(steps)]
        e1.record(stream)
        barrier()
        t_end = time.monotonic()
        ms = e0.elapsed_time(e1)
        clocks = sampler.window(t_begin, t_end) if rank == 0 else None
        if dist is not None:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, B.kernel_launches() - launches0, clocks, extra

    hbm_peak, peak_src = peaks()
    if args.workload in ("search", "gather"):
        r = bench_search_gather(args, torch, dist, B, rank, world, timed, args.workload)
        if rank == 0:
            r.update({"n_gpus": world, "steps": args.steps, "warmup": args.warmup, "data": "synthetic", "dtype": "u64"})
            emit_json(r)
        if args.dump_outputs:
            write_outputs(args.dump_outputs)
        if dist is not None:
            dist.destroy_process_group()
        return
    out = {}
    if args.workload in ("compare", "both"):
        out["compare"] = bench_compare(args, torch, dist, B, rank, world, timed, hbm_peak, peak_src)
    if args.workload in ("sketch", "both"):
        out["sketch"] = bench_sketch(args, torch, dist, B, rank, world, timed, hbm_peak, peak_src)
    if rank == 0:
        primary = out.get("compare") or out.get("sketch")
        line = dict(primary)
        if "compare" in out and "sketch" in out:
            line["sketch"] = out["sketch"]
        emit_json(line)
    if args.dump_outputs:
        write_outputs(args.dump_outputs)
    if dist is not None:
        dist.destroy_process_group()


def bench_compare(args, torch, dist, B, rank, world, timed, hbm_peak, peak_src):
    h, off = compare_workload()
    n = len(off) - 1
    n_pairs = n * (n - 1) // 2
    sizes = np.diff(off.astype(np.int64))
    # algorithmic bytes of the intersection kernel: every pair reads both rows once, writes a u32
    alg_bytes = 8.0 * (n - 1) * float(sizes.sum()) + 4.0 * n_pairs
    dev = torch.device("cuda")
    B.set_profiling(True)

    if world == 1:
        sset = B.SketchSet.from_host(h, off)
        d_out = torch.empty((n, n), dtype=torch.float64, device=dev)
        kernel_ms = []

        def step():
            B.compare_jaccard_device(sset, d_out.data_ptr())

        def step_prof():
            step()
            kernel_ms.append(B.last_kernel_ms(0))

        ms, launches, clocks, _ = timed(step_prof, args.steps, args.warmup)
        kernel_ms = kernel_ms[-args.steps:]
        if args.dump_outputs:
            # the whole 10000 x 10000 matrix is 800 MB: a fixed, seeded choice of whole rows of it
            rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(n, 256), replace=False))
            keep_output("compare_jaccard_rows", d_out[torch.from_numpy(rows).to(dev)].cpu().numpy())
            keep_output("compare_jaccard_row_ids", rows.astype(np.float64))
        # end to end: host CSR (pinned) -> H2D -> kernels -> D2H of the float64 matrix (pinned)
        ph, po = B.pinned_empty(len(h), np.uint64), B.pinned_empty(len(off), np.uint64)
        ph.array[:] = h
        po.array[:] = off
        pout = B.pinned_empty((n, n), np.float64)

        def step_e2e():
            s2 = B.SketchSet.from_host(ph.array, po.array)
            B.compare_jaccard(s2, out=pout.array)
            return float(pout.array[0, 1])

        ms_e2e, _, _, _ = timed(step_e2e, max(2, args.steps // 2), 1)
        h2d, d2h = int(h.nbytes + off.nbytes), int(n * n * 8)
        parallelism = "1 gpu"
    else:
        # shard rows across ranks as if each rank had sketched its own genomes; one all-gather
        # of the shards, cyclic row tiles per rank, all-reduce of the partial count matrices,
        # each rank finalises a block of rows.
        from sourmash_b200.distributed import CompareShard
        cs = CompareShard(torch, dist, B, h, off, rank, world)
        kernel_ms = []

        def step_prof():
            cs.step(e2e=False)
            kernel_ms.append(B.last_kernel_ms(0))

        ms, launches, clocks, _ = timed(step_prof, args.steps, args.warmup)
        kernel_ms = kernel_ms[-args.steps:]
        ms_e2e, _, _, _ = timed(lambda: cs.step(e2e=True), max(2, args.steps // 2), 1)
        h2d, d2h = cs.h2d_bytes, cs.d2h_bytes
        alg_bytes = alg_bytes / world
        parallelism = (f"{world} gpus: sketches all-gathered, hash space split into {world} key ranges (sort + tags + whole-row "
                       "counting of one range per rank), partial counters reduce-scattered by row block, rows finalised per rank")

    value = n_pairs / (ms / 1e3)
    kms = float(np.mean(kernel_ms))
    achieved = alg_bytes / (kms / 1e3) / 1e9
    plan = B.last_compare_plan()
    if plan["algo"] == "join":
        knote = ("counts by sorting the hashes of the set once and incrementing one counter per pair of rows sharing a hash "
                 "(planner estimate: %.3g increments over %.3g elements); algorithmic bytes keep SURVEY 8d's "
                 "definition, 8*(|A|+|B|) per pair + 4 B out" % (plan["est_increments"], plan["est_elements"]))
        if os.environ.get("SMB_JOIN_LAYOUT", "") == "plain":      # A/B runs only: the global-reduction join
            kname = "inverted join, global reductions (join_gather + cub::DeviceRadixSort + join_count_kernel)"
            tkey = "inverted_join"
            plan = dict(plan, layout="plain")
        else:
            kname = ("inverted join, stripe layout (stripe_keys + cub::DeviceRadixSort on 32-bit keys + stripe_tag + "
                     "join_stripe_kernel + stripe_mirror; counters in shared memory, no global atomics)")
            tkey = "inverted_join_stripe"
            plan = dict(plan, layout=os.environ.get("SMB_JOIN_LAYOUT") or "stripe")
    else:
        kname, tkey = "pairwise_tile_split_kernel", "pairwise_tile_split_kernel"
        knote = ("algorithmic bytes = 8*(|A|+|B|) per pair + 4 B out; rows are reused from shared "
                 "memory / L2, so DRAM traffic is far below this")
    res = {
        "metric": "sketch-pairs/sec (compare)", "value": value, "unit": "pairs/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": COMPARE_WORKLOAD,
                   "n_sketches": n, "pairs_per_step": n_pairs, "parallelism": parallelism,
                   "l2_policy": "inputs 400 MB + 800 MB output per step exceed the 126 MB L2; no flush"},
        "e2e": {"value": n_pairs / (ms_e2e / 1e3), "unit": "pairs/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"kernel": kname, "bound": "hbm", "achieved": achieved, "peak": hbm_peak,
                     "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": ncu_traffic(tkey) if world == 1 else None,
                     "kernel_ms": kms, "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                     "algorithm": plan, "note": knote},
    }
    traffic = res["roofline"]["traffic"]
    if traffic:                                           # what actually crossed the HBM interface (ncu), same launches
        res["roofline"]["dram"] = {"bytes_per_launch": traffic, "achieved": traffic / world / (kms / 1e3) / 1e9,
                                   "unit": "GB/s", "frac": traffic / world / (kms / 1e3) / 1e9 / hbm_peak}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:      # CPU baseline: rank 0 at N=1 only
        ncores = host_cores()
        units, dt, sample, want = cpu_compare_sample(h, off, ncores, int(1.5e5 * ncores))
        res["cpu_baseline"] = {"value": units / dt, "unit": "pairs/s", "cores": ncores, "kind": "port",
                               "sample": sample, "seconds": dt}
        # the rows the CPU arm just computed are the parity check of the GPU matrix (resident path and end-to-end path):
        # float64 bit for bit, |delta| = 0 <= the 1e-12 of north_star
        nr = len(want)
        got_dev = d_out[:nr].cpu().numpy()
        iu = np.triu_indices(nr, 1, n)
        assert np.array_equal(got_dev[iu], want[iu]), "compare: GPU matrix differs from the CPU oracle rows"
        assert np.array_equal(pout.array[:nr][iu], want[iu]), "compare e2e: GPU matrix differs from the CPU oracle rows"
        assert np.array_equal(got_dev, pout.array[:nr]) and bool((np.diagonal(got_dev) == 1.0).all())
        assert np.array_equal(pout.array, pout.array.T), "compare: matrix not symmetric"
        res["parity_checked_pairs"] = int(units)
    return res


def bench_sketch(args, torch, dist, B, rank, world, timed, hbm_peak, peak_src):
    seqs, offs = sketch_workload()
    ng = len(offs) - 1
    mine = list(range(rank, ng, world))                   # genomes dealt round-robin to ranks
    my_off = np.zeros(len(mine) + 1, dtype=np.uint64)
    my_off[1:] = np.cumsum([int(offs[g + 1] - offs[g]) for g in mine])
    my_seqs = np.concatenate([seqs[int(offs[g]):int(offs[g + 1])] for g in mine]) if world > 1 else seqs
    total_kmers = sum(int(offs[g + 1] - offs[g]) - k + 1 for g in range(ng) for k in KSIZES)
    my_kmers = sum(int(offs[g + 1] - offs[g]) - k + 1 for g in mine for k in KSIZES)
    dev = torch.device("cuda")
    d_bases = torch.empty(len(my_seqs) + 64, dtype=torch.uint8, device=dev)
    d_bases[: len(my_seqs)].copy_(torch.from_numpy(my_seqs))
    lens = np.diff(my_off.astype(np.int64)).astype(np.uint64)
    B.set_profiling(True)
    kernel_ms = []

    gather_cache = {}

    def gather_shards(sset):
        if dist is None:
            return
        from sourmash_b200.distributed import allgather_sketchset
        allgather_sketchset(torch, dist, B, sset, cache=gather_cache)

    last = {}

    def step():
        sset, nk = B.sketch_streams_device(d_bases.data_ptr(), my_off[:-1], lens, KSIZES, scaled=SCALED)
        assert nk == my_kmers
        kernel_ms.append(B.last_kernel_ms(1))
        gather_shards(sset)
        last["sset"] = sset
        return None

    ms, launches, clocks, _ = timed(step, args.steps, args.warmup)
    kernel_ms = kernel_ms[-args.steps:]
    if args.dump_outputs:
        # one sketch per (genome, k), genome-major: ~1.5e6 hashes in all
        hh, oo = last["sset"].to_host()
        u64_as_float64("sketch_hashes", hh)
        keep_output("sketch_offsets", np.asarray(oo, dtype=np.float64))
    pin = B.pinned_empty(len(my_seqs), np.uint8)
    pin.array[:] = my_seqs

    def step_e2e():
        sset, nk = B.sketch_sequences(pin.array, my_off, KSIZES, scaled=SCALED)
        gather_shards(sset)
        hh, oo = sset.to_host()
        return int(oo[-1])

    ms_e2e, _, _, ex = timed(step_e2e, max(2, args.steps // 2), 1)
    kms = float(np.mean(kernel_ms))
    alg_bytes = float(my_kmers) * (1.0 + 8.0 / SCALED)
    achieved = alg_bytes / (kms / 1e3) / 1e9
    res = {
        "metric": "k-mers hashed/sec (sketch)", "value": total_kmers / (ms / 1e3), "unit": "k-mers/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": SKETCH_WORKLOAD,
                   "kmers_per_step": total_kmers,
                   "parallelism": "1 gpu" if world == 1 else f"{world} gpus: genomes round-robin, sketches all-gathered",
                   "l2_policy": "500 MB of bases per pass exceed the 126 MB L2; no flush"},
        "e2e": {"value": total_kmers / (ms_e2e / 1e3), "unit": "k-mers/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(len(my_seqs)), "d2h_bytes_per_step": int(ex[-1]) * 8},
        "gpu_launches": launches, "clocks": clocks,
        "roofline": {"kernel": "hash_kmers_kernel (3 launches, k=21,31,51)", "bound": "hbm", "achieved": achieved,
                     "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                     "traffic": ncu_traffic("hash_kmers_kernel"), "kernel_ms": kms,
                     "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                     "note": "integer-issue bound by construction (~150 int ops per k-mer vs 1 B): "
                             "HBM fraction is expected to be small; roofline.issue is the bound that applies"},
    }
    fused = os.environ.get("SMB_SKETCH_FUSED") != "0"      # default: k=21,31,51 in one pass; =0: three launches (A/B runs)
    if fused:
        res["roofline"]["kernel"] = "hash_kmers_fused_kernel (1 launch, k=21,31,51)"
        res["roofline"]["traffic"] = ncu_traffic("hash_kmers_fused_kernel")
    wipk = ncu_traffic("hash_kmers_fused_kernel_warp_instr_per_kmer" if fused else "hash_kmers_kernel_warp_instr_per_kmer")
    if wipk:
        # the bound that applies: warp instructions issued (ncu count of the same three launches, per k-mer)
        # against 4 issue slots per SM per clock at the SM clock sampled during the timed region
        clk = float((clocks or {}).get("sm_mhz") or 1965.0) * 1e6
        issued = wipk * my_kmers / (kms / 1e3)
        res["roofline"]["issue"] = {"warp_instructions_per_kmer": wipk, "achieved": issued / 1e9,
                                    "peak": SM_COUNT * 4 * clk / 1e9, "unit": "G warp-instr/s",
                                    "frac": issued / (SM_COUNT * 4 * clk),
                                    "source": ncu_source("hash_kmers_fused_kernel_warp_instr_per_kmer" if fused else "hash_kmers_kernel_warp_instr_per_kmer")}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ncores = host_cores()
        units, dt, sample, want = cpu_sketch_sample(seqs, offs, ncores, ng)
        res["cpu_baseline"] = {"value": units / dt, "unit": "k-mers/s", "cores": ncores, "kind": "port",
                               "sample": sample, "seconds": dt}
        # the sketches the CPU arm just produced are the parity check: identical hash sets, genome by genome and ksize by ksize
        rows = last["sset"].rows()
        for g in range(ng):
            for ki, k in enumerate(KSIZES):
                assert np.array_equal(rows[g * len(KSIZES) + ki], want[k][g]), ("sketch differs from the CPU oracle", g, k)
        res["parity_checked_sketches"] = ng * len(KSIZES)
        # SURVEY 8d config-2 variants (src/core/benches/compute.rs:27-31): B = every 89th base an N (windows holding it are
        # skipped), C = lower case (upper-cased by the kernel).  Timed like the clean input, checked on the first genomes.
        import oracle as orc
        res["variants"] = {}
        n_check = min(3, ng)
        for name, make in (("B: every 89th base N", lambda a: _with_n(a, 89)), ("C: lower case", lambda a: a | np.uint8(0x20))):
            v = make(seqs)
            d_bases[: len(v)].copy_(torch.from_numpy(v))
            vres = {}

            def vstep():
                vres["sset"], nk = B.sketch_streams_device(d_bases.data_ptr(), my_off[:-1], lens, KSIZES, scaled=SCALED)
                vres["ms"] = B.last_kernel_ms(1)
            vms, _, _, _ = timed(vstep, args.steps, args.warmup)
            vrows = vres["sset"].rows()
            mx = orc.max_hash_for_scaled(SCALED)
            for g in range(n_check):
                gseq = v[int(offs[g]):int(offs[g + 1])]
                for ki, k in enumerate(KSIZES):
                    assert np.array_equal(vrows[g * len(KSIZES) + ki], orc.sketch_scaled(gseq, k, mx)), (name, g, k)
            res["variants"][name] = {"ms_per_step": vms, "hash_kernel_ms": vres["ms"], "value": total_kmers / (vms / 1e3),
                                     "unit": "k-mer windows/s", "parity_checked_sketches": n_check * len(KSIZES)}
        d_bases[: len(my_seqs)].copy_(torch.from_numpy(my_seqs))
    return res


def _with_n(seq, every):
    out = seq.copy()
    out[every - 1::every] = ord("N")
    return out


def _maybe_index(args, B, db):
    """--index: build the inverted index of the resident database once, outside the timed region (it
    belongs to loading the database, like the upload); the build time is reported beside the result."""
    if not getattr(args, "index", False):
        return {}
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n_keys = db.build_index()
    torch.cuda.synchronize()
    return {"index": {"distinct_hashes": int(n_keys), "build_ms": (time.perf_counter() - t0) * 1e3,
                      "note": "inverted index (hash -> rows) of the resident database, built once at load"}}


DB_BACKEND = "torch"            # "numpy": rows drawn on the host (tiny dry runs without a CUDA torch)
DB_BLOCK_ROWS = 6250            # rows per generated block; shard bounds of 1/2/4/8 ranks fall on block borders


def build_database(torch, B, sizes, frac, query, seed, lo, hi, overrides=None):
    """Rows [lo, hi) of a synthetic database (sourmash_b200.synth.database_block) resident in HBM as a SketchSet.
    Returns (SketchSet, device tensor of the hashes or None, host offsets)."""
    from sourmash_b200.synth import database_block
    assert lo % DB_BLOCK_ROWS == 0 or lo == hi, "shards start on block borders"
    h_off = np.zeros(hi - lo + 1, dtype=np.uint64)
    h_off[1:] = np.cumsum(sizes[lo:hi])
    if DB_BACKEND == "numpy":
        parts = [database_block(sizes, frac, query, b, min(b + DB_BLOCK_ROWS, hi), seed, overrides=overrides)
                 for b in range(lo, hi, DB_BLOCK_ROWS)]
        hh = np.concatenate(parts) if parts else np.zeros(0, np.uint64)
        return B.SketchSet.from_host(hh, h_off), None, h_off
    dev = torch.device("cuda")
    d_h = torch.empty(max(int(h_off[-1]), 1), dtype=torch.int64, device=dev)
    qd = torch.from_numpy(np.asarray(query, dtype=np.uint64).view(np.int64)).to(dev)
    for b in range(lo, hi, DB_BLOCK_ROWS):
        e = min(b + DB_BLOCK_ROWS, hi)
        d_h[int(h_off[b - lo]):int(h_off[e - lo])] = database_block(sizes, frac, qd, b, e, seed, overrides=overrides,
                                                                    torch=torch, device=dev)
    d_off = torch.from_numpy(h_off.view(np.int64)).to(dev)
    return B.SketchSet.from_device(d_h.data_ptr(), d_off.data_ptr(), h_off, keepalive=(d_h, d_off)), d_h, h_off


def _rows_to_host(torch, sset, d_h, h_off, n_rows):
    "the first n_rows rows of a database as host CSR (for the CPU checker)"
    n_rows = min(n_rows, len(h_off) - 1)
    end = int(h_off[n_rows])
    if d_h is None:
        hh, _ = sset.to_host()
        return hh[:end], h_off[: n_rows + 1]
    return d_h[:end].cpu().numpy().view(np.uint64), h_off[: n_rows + 1]


SEARCH_WORKLOAD = ("configs[3]: 1 query of 1e7 hashes uniform in [1, max_hash(1000)] vs a resident database of 300000 "
                   "sketches (~5000 hashes each, 12 GB; 1 % of the subjects draw 20-80 % of their hashes from the query), "
                   "|query ∩ subject| for every subject")
GATHER_WORKLOAD = ("configs[4]: gather of a ~1e5-hash metagenome query vs a resident database of 50000 sketches (2 GB), 200 of "
                   "them planted in 20 overlapping clusters, threshold 50 hashes")


def bench_search_gather(args, torch, dist, B, rank, world, timed, which):
    """configs[3] / configs[4] (SURVEY 8d): one query against a large resident database.  Rows are sharded by
    subject over the ranks (SURVEY 8e): search = local counts + one all-gather of the counters; gather = the
    session rounds with (best count, row) all-gathered and the winner's intersection broadcast."""
    from sourmash_b200.synth import database_plan, gather_workload, search_query
    from sourmash_b200.distributed import shard_bounds
    hbm_peak, peak_src = peaks()
    if which == "search":
        n_db = N_DB_SEARCH
        query = search_query(N_QUERY_SEARCH)
        sizes, frac = database_plan(n_db, 4001, planted_frac=0.01)
        overrides = None
    else:
        n_db = N_DB_GATHER
        query, sizes, frac, overrides = gather_workload(n_db)
    bounds = shard_bounds(n_db, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    t0 = time.time()
    db, d_h, h_off = build_database(torch, B, sizes, frac, query, 4002 if which == "search" else 5002, lo, hi, overrides)
    log(f"[bench] {which} database: rows [{lo}, {hi}) = {int(h_off[-1])} hashes resident ({time.time() - t0:.1f}s)")
    index_info = _maybe_index(args, B, db)
    n_hashes_total = int(sizes.sum())
    parallelism = "1 gpu" if world == 1 else "%d gpus: database sharded by subject, query replicated" % world
    if which == "search":
        return _bench_search(args, torch, dist, B, rank, world, timed, query, db, d_h, h_off, lo, hi, n_db, n_hashes_total,
                             hbm_peak, peak_src, parallelism, index_info)
    return _bench_gather(args, torch, dist, B, rank, world, timed, query, db, d_h, h_off, lo, hi, n_db, overrides,
                         parallelism, index_info)


def shard_bounds_of(n, world):
    from sourmash_b200.distributed import shard_bounds
    return shard_bounds(n, world)


def _bench_search(args, torch, dist, B, rank, world, timed, query, db, d_h, h_off, lo, hi, n_db, n_hashes_total, hbm_peak,
                  peak_src, parallelism, index_info):
    dev = torch.device("cuda")
    nq = len(query)
    d_q = torch.from_numpy(query.view(np.int64)).to(dev)
    d_counts = torch.zeros(max(hi - lo, 1), dtype=torch.int32, device=dev)
    pq = B.pinned_empty(nq, np.uint64)
    pq.array[:] = query
    if world == 1:
        def step():
            B.one_vs_many_device(d_q.data_ptr(), nq, db, d_counts.data_ptr())

        def step_e2e():
            return int(B.one_vs_many(pq.array, db).sum())
        gathered = None
    else:
        from sourmash_b200.distributed import ShardedDatabase
        sdb = ShardedDatabase(torch, dist, B, db, n_db, lo)
        per = max(b1 - b0 for b0, b1 in zip(shard_bounds_of(n_db, world)[:-1], shard_bounds_of(n_db, world)[1:]))
        d_counts = torch.zeros(per, dtype=torch.int32, device=dev)
        d_all = torch.zeros(per * world, dtype=torch.int32, device=dev)

        def step():
            sdb.search_counts_device(d_q, d_counts, d_all)

        def step_e2e():
            return int(sdb.search_counts(pq.array).sum())
    ms, launches, clocks, _ = timed(step, args.steps, args.warmup)
    if args.dump_outputs:
        keep_output("search_counts", d_counts[: hi - lo].cpu().numpy().astype(np.float64))
    ms_e2e, _, _, ex = timed(step_e2e, max(2, args.steps // 2), 1)
    alg = 8.0 * (n_hashes_total + nq * world)                    # every database hash once; the query once per rank
    achieved = alg / (ms / 1e3) / 1e9
    res = {"metric": "subjects searched/sec (search: 1e7-hash query vs 300000-sketch database)", "value": n_db / (ms / 1e3),
           "unit": "subjects/s", "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "config": {"workload": SEARCH_WORKLOAD, "db_hashes": n_hashes_total, "query_hashes": nq, "parallelism": parallelism,
                      "l2_policy": "12 GB streamed per pass: far beyond the 126 MB L2; no flush"},
           "e2e": {"value": n_db / (ms_e2e / 1e3), "unit": "subjects/s", "ms_per_step": ms_e2e,
                   "h2d_bytes_per_step": int(query.nbytes), "d2h_bytes_per_step": int(4 * n_db)},
           "gpu_launches": launches, "clocks": clocks,
           "roofline": {"kernel": "inverted index probe (index_count_kernel)" if index_info else
                        ("one_vs_many_global_kernel" if os.environ.get("SMB_SEARCH_LAYOUT") == "global" else
                         "one_vs_many_range_major_kernel (streams the range-major copy of the database)"),
                        "bound": "hbm", "achieved": achieved, "peak": hbm_peak * world, "unit": "GB/s",
                        "frac": achieved / (hbm_peak * world), "kernel_ms": ms,
                        "traffic": ncu_traffic("one_vs_many_range_major_kernel")
                        if world == 1 and not index_info and os.environ.get("SMB_SEARCH_LAYOUT") != "global" else None,
                        "algorithmic_bytes_per_launch": alg, "peak_source": peak_src,
                        "note": "whole pass timed (query and database resident): kernel_ms == ms_per_step"},
           **index_info}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # CPU arm on a bounded sample: the reference's walk (count_common per subject) over the first rows; its counts
        # are also the parity check of the GPU counters for those rows
        import oracle as orc
        all_host_cpus()
        ncores = host_cores()
        n_sample = min(hi - lo, 60 * ncores)
        hh, oo = _rows_to_host(torch, db, d_h, h_off, n_sample)
        t = time.perf_counter()
        want = orc.one_vs_many(query, hh, oo, nthreads=ncores)
        dt = time.perf_counter() - t
        got = d_counts[:n_sample].cpu().numpy()
        assert np.array_equal(got.astype(np.uint64), want), "search counters differ from the CPU oracle"
        res["cpu_baseline"] = {"value": n_sample / dt, "unit": "subjects/s", "cores": ncores, "kind": "port", "seconds": dt,
                               "sample": "the first %d subjects of the database, the whole query" % n_sample}
        res["parity_checked_subjects"] = int(n_sample)
    return res


def _gather_on_host(query, rows, threshold):
    """CounterGather rounds on the CPU (index/__init__.py:777-909, search.py:877-949) over candidate rows given as
    {row id: hashes}: pick the largest remaining overlap (lowest row id on ties), subtract its intersection."""
    import oracle as orc
    ids = sorted(rows)
    q = np.asarray(query, dtype=np.uint64)
    counts = {j: int(orc.count_common(q, rows[j])) for j in ids}
    picks = []
    while True:
        live = [j for j in ids if counts[j] >= max(threshold, 1)]
        if not live:
            break
        best = max(counts[j] for j in live)
        j = min(x for x in live if counts[x] == best)
        isect = np.intersect1d(q, rows[j])
        picks.append((j, len(isect)))
        for x in ids:
            if counts[x]:
                counts[x] -= int(orc.count_common(isect, rows[x]))
        q = np.setdiff1d(q, isect)
        if not len(q):
            break
    return picks


def _bench_gather(args, torch, dist, B, rank, world, timed, query, db, d_h, h_off, lo, hi, n_db, overrides, parallelism,
                  index_info):
    res = {}
    if world == 1:
        def step():
            ids, sizes = B.gather(query, db, threshold=50)
            res["picks"] = (ids, sizes)
            return len(ids)
    else:
        from sourmash_b200.distributed import ShardedDatabase
        sdb = ShardedDatabase(torch, dist, B, db, n_db, lo)

        def step():
            ids, sizes = sdb.gather(query, threshold=50)
            res["picks"] = (ids, sizes)
            return len(ids)
    ms, launches, clocks, ex = timed(step, args.steps, args.warmup)
    ids, isizes = res["picks"]
    if args.dump_outputs:
        keep_output("gather_rows", np.asarray(ids, dtype=np.float64))
        keep_output("gather_intersect_sizes", np.asarray(isizes, dtype=np.float64))
    out = {"metric": "gather wall time (configs[4])", "value": ms, "unit": "ms", "higher_is_better": False, "ms_per_step": ms,
           "scaling": "strong", "vs_baseline": None,
           "config": {"workload": GATHER_WORKLOAD, "query_hashes": int(len(query)), "db_rows": n_db, "parallelism": parallelism},
           "e2e": {"value": ms, "unit": "ms", "ms_per_step": ms, "h2d_bytes_per_step": int(query.nbytes),
                   "d2h_bytes_per_step": int(8 * len(ids)),
                   "note": "the query comes from host memory and the picks go back every step: the timed call is the end-to-end call"},
           "rounds": int(len(ids)), "rounds_per_s": len(ids) / (ms / 1e3), "gpu_launches": launches, "clocks": clocks,
           **index_info}
    if rank == 0 and not args.no_cpu_baseline:
        # only planted rows can reach the threshold (a random row shares ~0 hashes with the query): the CPU rounds run
        # over them; equality of the pick list (rows and intersection sizes, in order) is the parity check
        all_host_cpus()
        t = time.perf_counter()
        want = _gather_on_host(query, overrides, 50)
        dt = time.perf_counter() - t
        got = list(zip((int(x) for x in ids), (int(x) for x in isizes)))
        assert got == want, "gather picks differ from the CPU rounds: %r vs %r" % (got[:5], want[:5])
        out["cpu_baseline"] = {"value": dt * 1e3, "unit": "ms", "cores": 1, "kind": "port", "seconds": dt,
                               "sample": "the rounds over the %d planted rows only (the prefetch pass over the other %d rows "
                                         "is not timed)" % (len(overrides), n_db - len(overrides))}
        out["parity_checked_rounds"] = len(want)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of each workload; the end-to-end legs (host buffers in and out) run "
                         "max(2, steps // 2) more")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=["compare", "sketch", "both", "search", "gather"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--index", action="store_true",
                    help="search / gather workloads: query through the inverted index of the resident database")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, save what the last timed step computed as DIR/<name>.npy "
                         "(float32/float64, at most 64 MB, a fixed seeded sample of larger outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs needs --impl b200 in a single process")
    if args.workload is None:
        args.workload = "compare" if args.impl == "reference" else "both"
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    protect_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
