#!/usr/bin/env python
"""bench.py — rows/s of the projection -> fp64->fp32 cast -> histogram hot path on B200.

Workloads (BASELINE.json ``configs``; SURVEY.md §8d):

* ``s100`` (default; configs[2] at N = 1, configs[3] at N > 1): synthetic columnar table, 100 000 000 rows x 32 fp64
  columns, K = 32 projected columns (a fixed permutation), fp32 output table written, 256-bin histogram of every
  projected column over [-1000, 1000].
* ``s10`` (configs[1]): 10 000 000 x 16 fp64, projection + fp32 cast only.
* ``m`` (configs[4]): MNIST-shaped 1 000 000 x 784 uint8 table, per-column 256-bin value counts.

With N GPUs (one rank per GPU, torchrun) the rows are range-sharded and every step's partial histograms are merged
by the library itself (``ShardedEngine`` -> ``lo_group_*``): in-kernel peer-memory merge over NVLink, or one NCCL
all-reduce (``--merge nccl``).  Strong scaling: the table size is fixed.  One "step" = one pass of the hot path over
the table, merge included.  After the timed region the merged counts and the fp32 output checksums of EVERY run are
compared with oracle-made goldens (tests/golden/bench_goldens.json); a mismatch fails the run (rc 3).

Output: ONE JSON line on rank 0.

    python bench.py                            # 1 GPU, s100
    python bench.py --workload m               # config M
    torchrun ... bench.py --gpus 8             # one rank per GPU
    python bench.py --impl reference           # CPU arm: the oracle port on all host cores
    python bench.py --dump-outputs DIR         # also write the last timed step's outputs as DIR/<name>.npy

The bench runs the native libraries that ``__graft_entry__.build()`` left in the tree and writes nothing into the tree,
so it also runs from a read-only checkout.
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
from pathlib import Path

import numpy as np

sys.dont_write_bytecode = True      # no __pycache__ next to the package sources
ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SEED = 20260921
GEN_LO, GEN_HI = -1000.0, 1000.0
NBINS = 256
GOLDENS = ROOT / "tests" / "golden" / "bench_goldens.json"
METRIC = "rows/sec project+cast+histogram 100M×32 fp64→fp32; HBM GB/s vs peak @1/2/4/8 GPU"   # BASELINE.json "metric"
try:
    METRIC = json.loads((ROOT / "BASELINE.json").read_text())["metric"]
except Exception:
    pass

WORKLOADS = {
    # name: (rows, cols, dtype label, algorithmic bytes per row per projected column)
    "s100": {"rows": 100_000_000, "cols": 32, "dtype": "f64->f32", "bytes_per_elem": 12.0,
             "kernel": "lo::k_project_cast_hist<1,true,true,true>"},
    "s10": {"rows": 10_000_000, "cols": 16, "dtype": "f64->f32", "bytes_per_elem": 12.0,
            "kernel": "lo::k_project_cast_hist<1,false,true,false>"},
    "m": {"rows": 1_000_000, "cols": 784, "dtype": "u8", "bytes_per_elem": 1.0, "kernel": "lo::k_hist_u8_cols_lanes<2>"},
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def projected_columns(ncols: int) -> list[int]:
    """K = C, a fixed non-identity permutation (SURVEY.md §8: 'all columns, arbitrary permutation')."""
    return [(7 * j + 3) % ncols for j in range(ncols)] if ncols % 7 else list(range(ncols))[::-1]


K_SELECT = 0      # --k: project only the first K columns of the permutation (SURVEY.md §8d's selective K = C/4 run)


def workload_columns(workload: str, ncols: int) -> list[int]:
    if workload == "m":
        return list(range(ncols))
    cols = projected_columns(ncols)
    return cols[:K_SELECT] if 0 < K_SELECT < ncols else cols


def peaks() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def workload_text(workload: str, rows: int, ncols: int, k: int) -> str:
    if workload == "m":
        return f"per-column 256-bin value counts, {rows} x {ncols} uint8 (MNIST-shaped), columnar"
    if workload == "s10":
        return f"projection + fp32 cast, {rows} x {ncols} fp64 -> fp32, K={k} ({'permutation' if k == ncols else 'selective'}), columnar"
    return (f"fused project+cast+{NBINS}-bin histogram, {rows} x {ncols} fp64 -> fp32, K={k} ({'permutation' if k == ncols else 'selective'}), columnar, "
            f"range [{GEN_LO}, {GEN_HI}]")


class ClockSampler:
    """SM clock / power / throttle reasons sampled DURING the timed region (B200_PROFILING.md 'clocks line').
    NVML is polled from a thread every ~2 ms (the timed region of an 8-GPU run lasts ~15 ms: `nvidia-smi -lms` cannot
    go below 100 ms and would see it once at best); `nvidia-smi -lms 100` is the fallback when NVML is not importable.
    Every sample is stamped on receipt and only those inside [mark_start, mark_end] are summarised."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, device: int):
        self.device, self.rows, self.proc, self.thread = device, [], None, None
        self.t0 = self.t1 = None
        self.source, self._stop, self._smax = None, threading.Event(), None

    def _physical_index(self) -> int:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.device])
            except Exception:
                pass
        return self.device

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self._physical_index())
            self._smax = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            masks = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons

            def poll():
                while not self._stop.is_set():
                    try:
                        sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                        pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                        bits = int(reasons_fn(h))
                        self.rows.append((time.time(), sm, pw, [n for n in self.NAMES if bits & masks[n]]))
                    except Exception:
                        pass
                    time.sleep(0.002)
            self.source = "nvml, 2 ms poll"
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.source = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.device), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.source = "nvidia-smi -lms 100"
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            try:
                self._smax = float(r[2])
                self.rows.append((time.time(), float(r[1]), float(r[3]),
                                  [n for n, v in zip(self.NAMES, r[5:9]) if v.lower().startswith("active")]))
            except Exception:
                continue

    def wait_ready(self, wait_s: float = 2.0):
        """Block until samples are actually arriving.  Must be called BEFORE the barrier that precedes the timed
        region: only rank 0 samples, and waiting after the barrier would let the other ranks start their timed steps
        and then sit in the merge waiting for rank 0."""
        deadline = time.time() + wait_s
        while self.source is not None and not self.rows and time.time() < deadline:
            time.sleep(0.01)

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self) -> dict:
        if self.source is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML and no nvidia-smi"]}
        time.sleep(0.01 if self.proc is None else 0.12)
        self._stop.set()
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        inside = [r for r in self.rows if self.t0 is not None and self.t0 <= r[0] <= (self.t1 or r[0])]
        used = inside if inside else self.rows[-3:]
        sm = [r[1] for r in used]
        reasons = sorted({n for r in used for n in r[3]})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                "sm_max_mhz": self._smax, "power_w_max": max((r[2] for r in used), default=None), "samples": len(used),
                "samples_inside_timed_region": len(inside), "reasons": reasons, "source": self.source}


# ======================================================================================================
# CPU arm: the oracle port (oracle/bsem.c, OpenMP, all host cores)
# ======================================================================================================
def _cpu_sample_rows(workload: str, rows: int, ncols: int, requested: int) -> int:
    """Rows of the CPU sample: the WHOLE table when the host has the memory for it (so the arm runs the same
    config), else a bounded prefix; ``--cpu-rows`` forces a size."""
    if requested:
        return min(rows, requested)
    import psutil
    per_row = ncols * (1 if workload == "m" else 12)
    fit = int(psutil.virtual_memory().available * 0.5 / per_row)
    return rows if fit >= rows else max(1_000_000, fit // 1_000_000 * 1_000_000)


def cpu_pass_setup(workload: str, sample_rows: int, ncols: int):
    """Builds the oracle, generates the sample with the same OpenMP team / static row partition that later scans it
    (parallel first touch: every page lives on the NUMA node of the thread that reads it), returns one_pass()."""
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    import ctypes as C
    from oracle import cport
    threads = cport.use_all_cores()
    L = cport.lib()
    cols = workload_columns(workload, ncols)
    k = len(cols)
    idx = np.ascontiguousarray(cols, dtype=np.int32)
    if workload == "m":
        ins = [np.empty(sample_rows, dtype=np.uint8) for _ in range(k)]
        in_p = (C.c_void_p * k)(*[a.ctypes.data for a in ins])
        L.oracle_synth_fill_u8_mt(C.c_uint64(SEED), idx.ctypes.data_as(C.c_void_p), C.c_int(k), C.c_int64(0),
                                  C.c_int64(sample_rows), in_p)
        counts = np.zeros((k, 256), dtype=np.uint64)

        def one_pass():
            L.oracle_hist_u8_cols(in_p, C.c_int64(sample_rows), C.c_int(k), counts.ctypes.data_as(C.c_void_p))
            return counts
        return one_pass, threads, (ins,)
    ins = [np.empty(sample_rows, dtype=np.float64) for _ in range(k)]
    outs = [np.empty(sample_rows, dtype=np.float32) for _ in range(k)]
    in_p = (C.c_void_p * k)(*[a.ctypes.data for a in ins])
    out_p = (C.c_void_p * k)(*[a.ctypes.data for a in outs])
    L.oracle_synth_fill_f64_mt(C.c_int(0), C.c_uint64(SEED), idx.ctypes.data_as(C.c_void_p), C.c_int(k), C.c_int64(0),
                               C.c_int64(sample_rows), C.c_double(GEN_LO), C.c_double(GEN_HI), in_p, out_p)
    nb = NBINS if workload == "s100" else 0
    lo = np.full(k, GEN_LO, np.float32)
    hi = np.full(k, GEN_HI, np.float32)
    counts = np.zeros((k, max(nb, 1)), dtype=np.uint64)

    def one_pass():
        L.oracle_project_cast_hist(in_p, C.c_int64(sample_rows), C.c_int(k), out_p, C.c_int(nb),
                                   lo.ctypes.data_as(C.c_void_p), hi.ctypes.data_as(C.c_void_p),
                                   counts.ctypes.data_as(C.c_void_p))
        return counts
    return one_pass, threads, (ins, outs)


def _host_info() -> dict:
    """What the CPU arm actually had: the pool's 1-GPU boxes are slices of a host (same 128 logical CPUs visible, a
    fraction of the machine behind them), the 8-GPU box is the whole machine — the arm's rows/s differs ~6x between
    them for that reason, not because of the code (VERDICT r1 weak #5)."""
    info = {"logical_cpus": os.cpu_count(), "affinity_cpus": len(os.sched_getaffinity(0))}
    for key, path in (("cgroup_cpu_max", "/sys/fs/cgroup/cpu.max"), ("loadavg", "/proc/loadavg")):
        try:
            info[key] = Path(path).read_text().strip()
        except Exception:
            pass
    try:
        import psutil
        info["ram_gb"] = round(psutil.virtual_memory().total / 2 ** 30)
    except Exception:
        pass
    return info


def _sample_text(workload, sample_rows, rows, ncols, threads):
    whole = "the whole table" if sample_rows == rows else f"the first {sample_rows} rows of the {rows}-row table"
    return (f"{whole} x {ncols} cols of the same synthetic data, host-resident columns generated and scanned by the "
            f"same {threads}-thread OpenMP team (static row partition, parallel first touch, OMP_PROC_BIND=close), "
            "oracle port oracle/bsem.c (gcc -O2 -fopenmp); the reference's own PySpark+MongoDB path cannot run here "
            "(no JVM / pyspark / pymongo / mongod)")


def run_cpu_baseline(workload: str, rows: int, ncols: int, requested_rows: int, budget_s: float = 25.0) -> dict:
    sample_rows = _cpu_sample_rows(workload, rows, ncols, requested_rows)
    one_pass, threads, _keep = cpu_pass_setup(workload, sample_rows, ncols)
    one_pass()
    times, t_all = [], time.perf_counter()
    while len(times) < 7 and (len(times) < 3 or time.perf_counter() - t_all < budget_s):
        t0 = time.perf_counter()
        one_pass()
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return {"value": sample_rows / med, "unit": "rows/s", "cores": threads, "kind": "port", "passes": len(times),
            "sample_rows": sample_rows, "same_config": sample_rows == rows, "host": _host_info(),
            "sample": _sample_text(workload, sample_rows, rows, ncols, threads) + f"; median of {len(times)} passes"}


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = args.workload
    ncols, rows = args.cols, args.rows
    sample_rows = _cpu_sample_rows(w, rows, ncols, args.cpu_rows)
    one_pass, threads, _keep = cpu_pass_setup(w, sample_rows, ncols)
    for _ in range(args.warmup):
        one_pass()
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        one_pass()
        times.append(time.perf_counter() - t0)
    dt = sum(times)
    value = sample_rows * args.steps / dt
    k = len(workload_columns(w, ncols))
    sample = _sample_text(w, sample_rows, rows, ncols, threads)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "ms_per_step_median": statistics.median(times) * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": WORKLOADS[w]["dtype"], "data": "synthetic",
        "config": {"workload": workload_text(w, rows, ncols, k), "name": w, "rows": rows, "cols": ncols, "k": k,
                   "nbins": NBINS if w != "s10" else 0, "sample_rows": sample_rows, "threads": threads,
                   "same_config": sample_rows == rows,
                   "note": "reference PySpark/MongoDB stack is not runnable offline; this is the CPU oracle port"},
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port", "sample": sample, "host": _host_info()},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


# ======================================================================================================
# executor level: the reference's three operator classes on an in-process collection
# ======================================================================================================
def run_executor_e2e(engine, rows: int, with_cpu: bool) -> dict:
    """rows/s through ``DataType.convert_existent_file`` ("number": text -> binary64 on the GPU),
    ``Histogram.create_file`` (exact value counts = the reference's $group; and the binned extension, cold then warm
    from the HBM-resident copy) and ``Projection.create`` (castTo float32), on a ``rows``-row collection held by the
    in-process columnar store — the call a user of the reference's classes makes, host documents in, host documents
    out.  ``reference_like``: the reference's own per-document algorithm (oracle/rsem.py restatement of
    data_type_update.py:15-45 and a Counter group-by) on a 200k-row sample, single thread as the reference runs it."""
    import pyarrow as pa
    import pyarrow.compute as pc
    from learningorchestra_b200 import utils
    from learningorchestra_b200.column_store import ColumnarDatabase, TextColumn
    from learningorchestra_b200.data_type_update import DataType
    from learningorchestra_b200.histogram import Histogram
    from learningorchestra_b200.projection import Projection

    rng = np.random.default_rng(SEED)
    t0 = time.perf_counter()
    fare = np.round(rng.uniform(0, 600, rows), 4)
    age = np.where(rng.random(rows) < 0.2, np.nan, np.round(rng.uniform(0, 90, rows), 1))
    pclass = rng.integers(1, 4, rows)
    sib = rng.integers(0, 9, rows)
    text = {
        "Fare": pc.cast(pa.array(fare), pa.large_string()),
        "Age": pc.fill_null(pc.cast(pa.array(age, from_pandas=True), pa.large_string()), ""),       # blanks, as the CSV has them
        "Pclass": pc.cast(pa.array(pclass), pa.large_string()),
        "SibSp": pc.cast(pa.array(sib), pa.large_string()),
        "Embarked": pa.array(np.array(["S", "C", "Q", ""])[rng.integers(0, 4, rows)], type=pa.large_string()),
    }
    db = ColumnarDatabase()
    db.ingest_columns("big", {k: TextColumn(v) for k, v in text.items()})
    build_s = time.perf_counter() - t0
    out = {"rows": rows, "store": "column_store.ColumnarDatabase (Arrow text columns, as POST /files leaves them)",
           "build_s": build_s}

    def timed(fn):
        a = time.perf_counter()
        fn()
        return time.perf_counter() - a

    def cast():
        job = DataType(db, utils.DataTypeMetadata(db), engine=engine)
        job.convert_existent_file("big", {"Fare": "number", "Age": "number", "Pclass": "number", "SibSp": "number"})
        job.wait(600)
    dt = timed(cast)
    out["datatype_number"] = {"fields": 4, "seconds": dt, "rows_per_s": rows / dt, "cells_per_s": 4 * rows / dt}

    def counts(name, fields):
        job = Histogram(db, utils.HistogramMetadata(db), engine=engine)
        job.create_file("big", name, list(fields))
        job.wait(600)
    dt = timed(lambda: counts("big_h1", ["Pclass", "Embarked", "Age"]))
    out["histogram_value_counts"] = {"fields": 3, "seconds": dt, "rows_per_s": rows / dt}

    def binned(name):
        job = Histogram(db, utils.HistogramMetadata(db), engine=engine)
        job.create_file("big", name, ["Fare", "Age", "Pclass", "SibSp"], bins=64)
        job.wait(600)
    dt_cold = timed(lambda: binned("big_b1"))
    dt_warm = timed(lambda: binned("big_b2"))
    out["histogram_binned"] = {"fields": 4, "bins": 64, "cold_seconds": dt_cold, "warm_seconds": dt_warm,
                               "cold_rows_per_s": rows / dt_cold, "warm_rows_per_s": rows / dt_warm,
                               "note": "cold builds the HBM-resident copy of the 4 columns; warm reuses it"}

    def project():
        job = Projection(utils.ProjectionMetadata(db), engine)
        job.create("big", "big_p", ["Fare", "Age"], "mongodb://h/database.big?r", "mongodb://h/database.big_p?r", cast_to="float32")
        job.wait(600)
    dt = timed(project)
    out["projection_cast_float32"] = {"fields": 2, "seconds": dt, "rows_per_s": rows / dt}
    meta = db.find_one("big_b2", {"_id": 0})
    out["finished_flags_ok"] = bool(meta and meta.get("finished")) and bool(db.find_one("big_p", {"_id": 0}).get("finished"))
    if with_cpu:
        from collections import Counter
        from oracle import rsem
        n = min(rows, 200_000)
        docs = [{"_id": i + 1, "Fare": a, "Age": b, "Pclass": c, "SibSp": d} for i, (a, b, c, d) in enumerate(zip(
            text["Fare"].slice(0, n).to_pylist(), text["Age"].slice(0, n).to_pylist(), text["Pclass"].slice(0, n).to_pylist(),
            text["SibSp"].slice(0, n).to_pylist()))]
        a = time.perf_counter()
        for f in ("Fare", "Age", "Pclass", "SibSp"):
            rsem.convert_field(docs, f, "number")
        dt = time.perf_counter() - a
        a = time.perf_counter()
        for f in ("Pclass", "Age"):
            Counter(d[f] for d in docs)
        dh = time.perf_counter() - a
        out["reference_like"] = {"sample_rows": n, "threads": 1, "datatype_number_rows_per_s": n / dt,
                                 "histogram_2_fields_rows_per_s": n / dh,
                                 "note": "oracle/rsem.py per-document loop over in-memory dicts; flatters the reference: no "
                                         "MongoDB round trip per document (data_type_update.py:45), no mongod $group scan"}
    return out


# ======================================================================================================
# GPU arm
# ======================================================================================================
def _claim_stdout() -> int:
    """The contract is ONE JSON line on stdout.  Libraries talk on fd 1 too (NCCL prints its version banner there
    when NCCL_DEBUG=VERSION is in the environment), so fd 1 is pointed at stderr for the whole run and the JSON line
    is written to a private duplicate of the real stdout at the end."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return real


def _emit(real_stdout: int, line: dict) -> None:
    os.write(real_stdout, (json.dumps(line) + "\n").encode())


def load_goldens(workload: str, rows: int, ncols: int):
    try:
        g = json.loads(GOLDENS.read_text())[workload]
    except Exception:
        return None
    if g["rows"] != rows or g["cols"] != ncols or g["seed"] != SEED:
        return None
    return g


DUMP_SAMPLE_BYTES = 32 << 20      # --dump-outputs: size of the sample of the fp32 output table


def dump_outputs(dump_dir: str, sh, out, k: int, nbins: int) -> list[Path]:
    """Writes what the last step handed its caller, as ``dump_dir/<name>.npy``, so that two builds can be compared
    output for output on identical inputs:

    * ``counts``: the merged ``k x nbins`` histogram, float64 (exact: every count is below 2^53);
    * ``out_f32_sample``: ``k x S`` float32, the same S rows of every projected output column, drawn without replacement
      by a generator seeded with SEED and kept in row order; S is what fits in DUMP_SAMPLE_BYTES.  The rows come from
      this rank's shard, which is the whole table on one GPU.
    """
    import torch
    arrays = {}
    if nbins:
        arrays["counts"] = sh.result(k * nbins).reshape(k, nbins).astype(np.float64)
    if out is not None:
        shard = out.shards[0]
        n = min(shard.nrows, DUMP_SAMPLE_BYTES // (4 * k))
        rows = torch.from_numpy(np.sort(np.random.default_rng(SEED).choice(shard.nrows, size=n, replace=False))).cuda()
        cols = [torch.as_tensor(shard.column_view(j), device="cuda")[rows] for j in range(k)]
        arrays["out_f32_sample"] = torch.stack(cols).cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > 64 * 10 ** 6:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed 64 MB")
    d = Path(dump_dir)
    d.mkdir(parents=True, exist_ok=True)
    paths = []
    for name, a in arrays.items():
        paths.append(d / f"{name}.npy")
        np.save(paths[-1], a)
    return paths


def run_gpu(args) -> int:
    real_stdout = _claim_stdout()
    import torch
    import torch.distributed as dist

    from learningorchestra_b200 import _native as N
    from learningorchestra_b200.engine import Engine
    from learningorchestra_b200.sharding import ShardedEngine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
        args.gpus = world
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    w = args.workload
    eng = Engine(local_rank)
    if world > 1:
        sh = ShardedEngine.from_torch_distributed(eng, merge={"p2p": "peer"}.get(args.merge, args.merge))
    else:
        sh = ShardedEngine.from_exchange(eng, 0, 1, lambda b: [b], lambda ok: ok, merge="peer")
    ncols, total_rows = args.cols, args.rows
    from learningorchestra_b200.engine import prepare_columns
    cols_list = workload_columns(w, ncols)
    k = len(cols_list)
    cols = prepare_columns(cols_list)        # converted once: 784 indices cost more Python time than config M's kernel
    # a non-default stream: libloexec launches on exactly the stream it is handed (NULL would mean its own), and
    # torch.cuda.Event then sees the same stream
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    streams = [stream]

    lo = np.full(k, GEN_LO, np.float32)
    hi = np.full(k, GEN_HI, np.float32)
    if w == "m":
        table = sh.table("u8", total_rows, ncols).fill_synthetic(N.LO_SYNTH_MNIST_U8, SEED, streams=streams)
        out = None
    else:
        table = sh.table("f64", total_rows, ncols).fill_synthetic(N.LO_SYNTH_UNIFORM, SEED, lo=GEN_LO, hi=GEN_HI, streams=streams)
        out = sh.table("f32", total_rows, k)
    nrows = table.local_rows
    torch.cuda.synchronize()

    kev = []   # (start, end) events around the library call of one ISOLATED step (no overlap with its neighbours)
    # Timed steps are independent jobs over the same resident table (each step re-reads its inputs and rewrites its
    # outputs; nothing is carried from step to step), so they are issued with LO_GROUP_INDEPENDENT: the next step's
    # CTAs may fill the SMs that the previous step's last wave leaves idle (programmatic dependent launch).  Every
    # step still does all of its work; --no-overlap serialises them completely, as round 1 did.
    overlap = not args.no_overlap

    def step(record: bool):
        if record:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
        ind = overlap and not record          # an event record between two launches serialises them anyway
        if w == "s100":
            sh.project_cast_hist(table, cols, NBINS, lo, hi, out=out, streams=streams, independent=ind)
        elif w == "s10":
            sh.project_cast(table, cols, out=out, streams=streams)
        else:
            sh.hist_u8_cols(table, cols, streams=streams, independent=ind)
        if record:
            e1.record(stream)
            kev.append((e0, e1))

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step(False)
    torch.cuda.synchronize()
    if sh.timeouts():
        raise SystemExit("a device-side wait of the merge timed out during warm-up")
    sampler.wait_ready()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.mark_start()
    launches0 = eng.launch_count
    # all GPUs enter the timed region together: a device-side barrier on the timing stream (a host barrier
    # leaves tens of microseconds of skew, which the root would then spend waiting inside step 0's merge)
    sh.barrier(streams)
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start.record(stream)
    for _ in range(args.steps):
        step(False)
    t_end.record(stream)
    torch.cuda.synchronize()
    sampler.mark_end()
    launches = eng.launch_count - launches0 - 1          # the barrier launch is outside the timed region
    if args.dump_outputs:
        if rank == 0:
            for p in dump_outputs(args.dump_outputs, sh, out, k, NBINS if w != "s10" else 0):
                log(f"wrote {p}")
        if world > 1:
            dist.barrier()                               # the merge of the next step waits for rank 0
    for _ in range(5):                                   # the same step in isolation (event-bracketed, serialised)
        step(True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    elapsed_ms = t_start.elapsed_time(t_end)
    kernel_ms = [a.elapsed_time(b) for a, b in kev]
    t = torch.tensor([elapsed_ms, sum(kernel_ms) / len(kernel_ms)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms, kernel_ms_isolated = float(t[0]), float(t[1])
    # average duration of the kernel over the timed region: one launch per step, back to back on one stream
    kernel_ms_avg = elapsed_ms / args.steps
    assert sh.timeouts() == 0, "a device-side wait of the merge timed out"

    # ---- parity of THIS run against the oracle-made goldens (every N, every workload) ---------------------
    gold = load_goldens(w, total_rows, ncols)
    parity = {"golden": str(GOLDENS.relative_to(ROOT)) if gold else None}
    final_counts = None
    if w != "s10" and sh.has_result:
        final_counts = sh.result(k * NBINS).reshape(k, NBINS)
    if out is not None:
        def as_i64(u: int) -> int:
            return u - (1 << 64) if u >= (1 << 63) else u
        sums = torch.tensor([as_i64(out.checksum(j)) for j in range(k)], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(sums)                     # two's-complement wrap == addition mod 2^64
        sums = [int(v) & 0xFFFFFFFFFFFFFFFF for v in sums.cpu().tolist()]
    if rank == 0:
        if final_counts is not None:
            total_counted = int(final_counts.sum())
            assert total_counted == total_rows * k, f"histogram lost rows: {total_counted} != {total_rows * k}"
        if gold is None:
            parity["note"] = "no golden for this rows / cols / seed; only the row-conservation check ran"
        else:
            if final_counts is not None:
                parity["counts"] = bool(np.array_equal(final_counts, np.array(gold["counts"], dtype=np.uint64).reshape(-1, NBINS)[:k]))
            if out is not None:
                parity["checksums"] = sums == [int(x) for x in gold["checksums"]][:k]
        parity["ok"] = all(v for kk, v in parity.items() if kk in ("counts", "checksums"))

    # ---- end to end: host buffers in, host buffers out, through the same group API ------------------------
    e2e, e2e_ready = None, False
    if not args.no_e2e:
        import psutil
        saved_affinity = os.sched_getaffinity(0)
        numa = None
        try:
            numa = eng.bind_numa()             # pinned buffers below are first touched next to this rank's GPU
        except Exception as exc:               # noqa: BLE001
            log(f"[rank {rank}] NUMA binding unavailable: {exc!r}")
        avail = psutil.virtual_memory().available
        per_row = (1 if w == "m" else 12) * k
        budget_rows = int(avail * 0.45 / world / per_row)
        e2e_rows = min(nrows, args.e2e_rows if args.e2e_rows else nrows, budget_rows)
        e2e_rows = max(61440, e2e_rows // 61440 * 61440) if e2e_rows >= 61440 else e2e_rows
        # set-up (pinned host buffers, staging) can fail on a box with little free RAM: every rank reports, and e2e
        # is skipped on ALL ranks together rather than leaving some of them waiting in a collective
        setup_error = None
        try:
            hin = eng.pinned_empty((k, e2e_rows), np.uint8 if w == "m" else np.float64, write_combined=args.e2e_wc)
            hout = eng.pinned_empty((k, e2e_rows), np.float32) if w != "m" else None
            for j in range(k):   # host inputs = the projected columns of this rank's shard (device -> pinned host, untimed)
                table.shards[0].to_numpy(cols_list[j], 0, e2e_rows, out=hin[j])
            in_cols = [hin[j] for j in range(k)]
            out_cols = [hout[j] for j in range(k)] if hout is not None else None

            def e2e_step():
                if w == "s100":
                    return sh.project_cast_hist_host(in_cols, NBINS, lo, hi, out=out_cols)
                if w == "s10":
                    return sh.project_cast_hist_host(in_cols, None, out=out_cols)
                return sh.hist_u8_cols_host(in_cols)
            e2e_step()                       # warm-up (allocates staging)
        except Exception as exc:          # noqa: BLE001
            setup_error = repr(exc)
            log(f"[rank {rank}] e2e set-up failed: {setup_error}")
        okf = torch.tensor([0.0 if setup_error else 1.0], device="cuda")
        if world > 1:
            dist.all_reduce(okf, op=dist.ReduceOp.MIN)
        e2e_ready = float(okf[0]) == 1.0
        if not e2e_ready:
            e2e = {"value": None, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                   "error": setup_error or "set-up failed on another rank"}
    if e2e_ready:
        if world > 1:
            dist.barrier()
        e2e_steps = max(1, min(args.steps, args.e2e_steps))
        l0 = eng.launch_count
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            c_host, tm = e2e_step()
        dt = time.perf_counter() - t0
        e2e_launches = eng.launch_count - l0
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        rr = torch.tensor([float(e2e_rows), tm["h2d_bytes"], tm["d2h_bytes"]], dtype=torch.float64, device="cuda")
        mn = torch.tensor([tm["h2d_bytes"] / dt * e2e_steps / 1e9], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(rr, op=dist.ReduceOp.SUM)
            dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        e2e_parity = None
        if rank == 0 and gold is not None and w != "s10" and int(float(rr[0])) == total_rows:
            e2e_parity = bool(np.array_equal(c_host, np.array(gold["counts"], dtype=np.uint64).reshape(-1, NBINS)[:k]))
        e2e = {"value": float(rr[0]) * e2e_steps / float(tt[0]), "unit": "rows/s",
               "h2d_bytes_per_step": int(float(rr[1])), "d2h_bytes_per_step": int(float(rr[2])),
               "rows_per_step": int(float(rr[0])), "steps": e2e_steps, "launches": e2e_launches,
               "h2d_GBs_slowest_rank": float(mn[0]), "numa": {"node": numa[0], "cpus": numa[1]} if numa else None,
               "counts_match_golden": e2e_parity,
               "api": ("ShardedEngine.hist_u8_cols_host -> lo_group_hist_u8_cols_host" if w == "m" else
                       "ShardedEngine.project_cast_hist_host -> lo_group_project_cast_hist_host")
                      + " (pinned host buffers, chunked H2D / kernel / D2H on three streams per GPU, equally strided "
                        "columns as one 2-D copy per chunk, counts merged over the group)"}
        os.sched_setaffinity(0, saved_affinity)

    rc = 0
    if rank == 0:
        peak, peak_src = peaks()
        W = WORKLOADS[w]
        alg_bytes = W["bytes_per_elem"] * k * nrows
        achieved = alg_bytes / (kernel_ms_avg * 1e-3) / 1e9
        cpu = run_cpu_baseline(w, total_rows, ncols, args.cpu_rows) if world == 1 and not args.no_cpu else None
        executor = None
        if world == 1 and w == "s100" and args.executor_rows > 0:
            try:
                table.free()
                if out is not None:
                    out.free()
                executor = run_executor_e2e(eng, args.executor_rows, not args.no_cpu)
            except Exception as exc:          # noqa: BLE001  (reported, never fatal for the headline line)
                executor = {"error": repr(exc)}
        gb_in = nrows * k * (1 if w == "m" else 8) / 1e9
        line = {
            "metric": METRIC, "value": total_rows * args.steps / (elapsed_ms * 1e-3), "unit": "rows/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps,
            "us_per_step": elapsed_ms / args.steps * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": W["dtype"],
            "data": "synthetic",
            "config": {"workload": workload_text(w, total_rows, ncols, k), "name": w,
                       "rows": total_rows, "cols": ncols, "k": k, "nbins": NBINS if w != "s10" else 0, "rows_per_gpu": nrows,
                       "merge": sh.merge if world > 1 else None, "steps_overlap": bool(overlap and w != "s10"),
                       "parallelism": (f"row-range shards x{world}, " + (
                           f"one NCCL all-reduce of {k}x{NBINS} uint64 per step (inside libloexec)" if sh.merge == "nccl" else
                           "merge inside the streaming kernel: column-last CTAs push with system-scope RED.64 into rank 0's "
                           "matrix over NVLink (CUDA IPC), arrival + root epilogue in-kernel, one launch per step"))
                                      if world > 1 else "single GPU",
                       "l2": (f"inputs larger than L2: {gb_in:.2f} GB read per GPU per step (L2 = 126 MB), no flush needed"
                              if gb_in > 0.5 else
                              f"{gb_in * 1e3:.0f} MB read per GPU per step: NOT larger than L2 (126 MB) at this N; "
                              "latency-dominated, reported in microseconds")},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "peak_source": peak_src, "kernel": W["kernel"],
                         "kernel_ms_avg": kernel_ms_avg, "algorithmic_bytes_per_launch": alg_bytes,
                         "kernel_ms_isolated": kernel_ms_isolated,
                         "note": ("kernel_ms_avg = timed region / steps (one launch per step, merge included"
                                  + (", consecutive launches allowed to overlap their predecessor's draining last wave" if overlap and w != "s10" else "")
                                  + "); kernel_ms_isolated = the same launch alone between two CUDA events, 5 samples after the timed region")},
            "parity": parity, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if executor:
            line["e2e_executor"] = executor
        tr = ROOT / "profiles" / "traffic.json"
        if tr.exists():
            try:
                key = {"s100": "k_project_cast_hist_bytes_per_launch", "m": "k_hist_u8_cols_bytes_per_launch"}.get(w)
                full = json.loads(tr.read_text()).get(key) if key else None      # ncu, one full-size launch
                line["roofline"]["traffic"] = full * nrows / W["rows"] if full else None
                line["roofline"]["traffic_source"] = ("ncu --set full dram__bytes_read+write of one full-size launch "
                                                      "(profiles/), scaled to this launch's rows")
            except Exception:
                pass
        _emit(real_stdout, line)
        if parity.get("ok") is False or (e2e and e2e.get("counts_match_golden") is False):
            log("PARITY FAILURE:", json.dumps(parity), json.dumps(e2e))
            rc = 3
    if world > 1:
        flag = torch.tensor([float(rc)], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        rc = int(flag[0])
        dist.barrier()
    sh.close()
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    return rc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="s100", choices=sorted(WORKLOADS))
    ap.add_argument("--rows", type=int, default=0)
    ap.add_argument("--cols", type=int, default=0)
    ap.add_argument("--k", type=int, default=0, help="project only the first K columns of the permutation (s100 / s10; 0 = all)")
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows of the CPU sample (0 = whole table when RAM allows)")
    ap.add_argument("--e2e-rows", type=int, default=0, help="cap on e2e rows per rank (0 = whole shard if RAM allows)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-wc", action="store_true", help="e2e input buffers in write-combined pinned memory (A/B knob)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--executor-rows", type=int, default=10_000_000,
                    help="rows of the in-process collection for the executor-level numbers (s100 at N = 1; 0 = skip)")
    ap.add_argument("--no-overlap", action="store_true",
                    help="serialise consecutive steps completely (no programmatic dependent launch between them)")
    ap.add_argument("--merge", default="auto", choices=["auto", "nccl", "p2p", "peer"],
                    help="N > 1: how partial histograms are merged (in-kernel peer-memory merge, or NCCL all-reduce)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm has none to write")
    args.rows = args.rows or WORKLOADS[args.workload]["rows"]
    args.cols = args.cols or WORKLOADS[args.workload]["cols"]
    global K_SELECT
    K_SELECT = max(0, args.k)
    if args.steps is None:
        args.steps = 100 if args.impl == "ours" else 5
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
        return 0
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
