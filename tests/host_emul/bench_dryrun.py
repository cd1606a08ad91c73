"""Dry run of bench.py's B200 arm without a GPU: the emulated library plays the device, a stand-in for the few
torch.cuda calls bench.py makes supplies streams / events / "device" tensors (host memory), and the workloads are
shrunk by patching bench's size constants from outside.  NOT a measurement -- it only proves that every code path of
bench.py assembles its JSON line (keys, types) without raising, for each workload and switch.
Run by tests/test_emulated_library.py.

    python tests/host_emul/bench_dryrun.py
"""
import io
import json
import os
import sys
import time
import types

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import emulated_boot  # noqa: E402

emulated_boot.install()

import torch  # noqa: E402


class _Stream:
    cuda_stream = 0

    def synchronize(self):
        pass


class _Event:
    def __init__(self, enable_timing=False):
        self.t = 0.0

    def record(self, stream=None):
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return max((other.t - self.t) * 1e3, 1e-3)


_real_empty, _real_zeros, _real_tensor = torch.empty, torch.zeros, torch.tensor


def _strip_device(fn):
    def wrapped(*a, **kw):
        kw.pop("device", None)
        return fn(*a, **kw)
    return wrapped


torch.empty, torch.zeros, torch.tensor = _strip_device(_real_empty), _strip_device(_real_zeros), _strip_device(_real_tensor)
torch.cuda.is_available = lambda: True
torch.cuda.set_device = lambda i: None
torch.cuda.current_stream = lambda *a: _Stream()
torch.cuda.synchronize = lambda *a: None
torch.cuda.Event = _Event
torch.cuda.current_device = lambda: 0
_real_device = torch.device
torch.Tensor.pin_memory = lambda self, *a, **kw: self

sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import bench  # noqa: E402

# tiny stand-ins for the two workload generators (the emulated device is ~10^4 x slower than a B200)
import numpy as np  # noqa: E402

from sourmash_b200.synth import synth_genome, synth_sketches  # noqa: E402


def _small_compare():
    return synth_sketches(160, mean=60, sd=15, lo=0, hi=120, n_families=5, pool=80, seed=1)


def _small_sketch(n_genomes=3):
    genomes = [synth_genome(12_000, seed=1000 + g) for g in range(3)]
    return np.concatenate(genomes), np.cumsum([0] + [len(g) for g in genomes]).astype(np.uint64)


bench.compare_workload, bench.sketch_workload = _small_compare, _small_sketch
bench.N_SKETCHES, bench.N_GENOMES, bench.GENOME_LEN = 160, 3, 12_000
# search / gather workloads: a 480-sketch database of ~60-hash rows, a 40 000-hash search query
import sourmash_b200.synth as _synth  # noqa: E402

_real_synth = _synth.synth_sketches
_synth.synth_sketches = lambda n, **kw: _real_synth(n, mean=60, sd=15, lo=10, hi=120, n_families=20, pool=80, seed=7)
bench.N_DB_SEARCH, bench.N_DB_GATHER, bench.N_QUERY_SEARCH = 480, 480, 40_000
bench.DB_BACKEND, bench.DB_BLOCK_ROWS = "numpy", 160      # rows drawn on the host
os.environ["SMB_RM_RANGES"] = "5"                         # few key ranges for the range-major copy of a tiny database
_real_plan, _real_gather = _synth.database_plan, _synth.gather_workload
_synth.database_plan = lambda n, seed, planted_frac=0.0, **kw: _real_plan(n, seed, planted_frac=max(planted_frac, 0.05) if planted_frac else 0.0,
                                                                         mean=60, sd=15, lo=10, hi=120)
_synth.gather_workload = lambda n_db, **kw: _real_gather(n_db, n_clusters=4, members=5, pool=70, noise=200)
_orig_device = torch.device
torch.device = lambda *a, **kw: _orig_device("cpu")

LINES = []
bench.emit_json = lambda obj: LINES.append(json.loads(json.dumps(obj)))


def run(workload, env=None, extra=(), cpu_baseline=False, dump_outputs=None):
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        args = types.SimpleNamespace(gpus=1, steps=1, warmup=3, impl="b200", workload=workload, no_cpu_baseline=not cpu_baseline,
                                     index="--index" in extra, dump_outputs=dump_outputs)
        bench._OUTPUTS.clear()
        n0 = len(LINES)
        bench.run_b200(args)
        assert len(LINES) == n0 + 1, "one JSON line per run"
        return LINES[-1]
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def main():
    base_keys = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                 "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"}
    line = run("both", {"SMB_COMPARE_ALGO": "join"}, cpu_baseline=True)      # with the CPU arm: its rows / sketches are the parity check
    assert line["parity_checked_pairs"] > 0 and line["sketch"]["parity_checked_sketches"] == 9
    assert len(line["sketch"]["variants"]) == 2 and all(v["parity_checked_sketches"] for v in line["sketch"]["variants"].values())
    assert base_keys <= set(line) and "sketch" in line and base_keys <= set(line["sketch"]), sorted(set(line))
    for part in (line, line["sketch"]):
        r = part["roofline"]
        assert {"kernel", "bound", "achieved", "peak", "unit", "frac", "traffic", "kernel_ms"} <= set(r)
        assert part["e2e"]["h2d_bytes_per_step"] > 0 and part["e2e"]["d2h_bytes_per_step"] > 0 and part["gpu_launches"] > 0
    # measured constants count only while the kernel files they were measured on are unchanged (profiles/ncu_traffic.json)
    assert ("dram" in line["roofline"]) == (line["roofline"]["traffic"] is not None)
    assert line["roofline"]["algorithm"]["algo"] == "join"
    for layout in ("stripe_full", "plain"):
        d = run("compare", {"SMB_COMPARE_ALGO": "join", "SMB_JOIN_LAYOUT": layout})
        assert d["roofline"]["algorithm"].get("layout") == layout
        assert ("stripe layout" in d["roofline"]["kernel"]) == (layout != "plain"), d["roofline"]["kernel"]
    d = run("compare", {"SMB_COMPARE_ALGO": "tile"})
    assert d["roofline"]["kernel"] == "pairwise_tile_split_kernel"
    assert "fused" in line["sketch"]["roofline"]["kernel"]
    d = run("sketch", {"SMB_SKETCH_FUSED": "0"})
    assert "3 launches" in d["roofline"]["kernel"]
    bench.N_SKETCHES = 240                                  # the tiled databases: 2 x 240 sketches
    for workload in ("search", "gather"):
        plain = run(workload, cpu_baseline=True)
        assert plain.get("parity_checked_subjects", 0) > 0 or plain.get("parity_checked_rounds", 0) > 0
        ranged = run(workload, {"SMB_SEARCH_LAYOUT": "global"})
        indexed = run(workload, extra=("--index",))
        assert {"metric", "value", "unit", "ms_per_step", "config", "gpu_launches", "n_gpus"} <= set(plain)
        assert "index" in indexed and indexed["index"]["distinct_hashes"] > 0 and "index" not in plain
        if workload == "gather":
            assert plain["rounds"] == ranged["rounds"] == indexed["rounds"] > 2, (plain["rounds"], ranged["rounds"], indexed["rounds"])
    # --dump-outputs: what the last timed step returned, float64 files, the same on a second run with the same arguments
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        for workload, names in (("both", {"compare_jaccard_rows", "compare_jaccard_row_ids", "sketch_hashes_hi32",
                                          "sketch_hashes_lo32", "sketch_offsets"}),
                                ("search", {"search_counts"}), ("gather", {"gather_rows", "gather_intersect_sizes"})):
            first, second = os.path.join(tmp, workload + "1"), os.path.join(tmp, workload + "2")
            run(workload, dump_outputs=first)
            run(workload, dump_outputs=second)
            assert set(os.listdir(first)) == {n + ".npy" for n in names}, sorted(os.listdir(first))
            for f in os.listdir(first):
                a, b = np.load(os.path.join(first, f)), np.load(os.path.join(second, f))
                assert a.dtype == np.float64 and a.size and np.array_equal(a, b), f
        rows = np.load(os.path.join(tmp, "both1", "compare_jaccard_rows.npy"))
        ids = np.load(os.path.join(tmp, "both1", "compare_jaccard_row_ids.npy")).astype(np.int64)
        assert rows.shape == (len(ids), len(_small_compare()[1]) - 1) and np.array_equal(rows[:, ids], rows[:, ids].T)
        hi, lo = (np.load(os.path.join(tmp, "both1", "sketch_hashes_%s32.npy" % p)).astype(np.uint64) for p in ("hi", "lo"))
        off = np.load(os.path.join(tmp, "both1", "sketch_offsets.npy")).astype(np.int64)
        hashes = (hi << np.uint64(32)) | lo
        assert len(off) == bench.N_GENOMES * len(bench.KSIZES) + 1 and off[-1] == len(hashes)
        from sourmash_b200.synth import MAX_HASH_1000
        assert len(hashes) and (hashes <= np.uint64(MAX_HASH_1000)).all()   # exact: the split keeps all 64 bits
    print("bench dry run ok: %d JSON lines assembled" % len(LINES))


if __name__ == "__main__":
    main()
