#!/usr/bin/env python3
"""bench.py — headline benchmark of the hot path (contract in the task prompt, SURVEY.md §8d).

Workload (BASELINE.json configs[1], C2): the numeric business-rules suite
    has_size, has_min(f0), has_mean(f1), has_correlation(f0, f1), satisfies("f2 > 0 AND i0 < 1000000")
on a synthetic 100 M-row x 8-column (4 f64 + 4 i64) table with 5 % nulls per column, per GPU
(row-partitioned, weak scaling). A "step" is one evaluation of the whole suite over one table.

    value      rows/s with the table already resident in HBM (adopted device buffers), whole job
    roofline   algorithmic bytes of the suite / average duration of the fused scan kernel (CUDA events
               recorded by the engine on its own stream around the launch) vs MEASURED_PEAKS.json hbm_gbs
    e2e        same metric through the public API from pinned HOST Arrow buffers: H2D staging of the
               referenced columns + scan + result read-back inside the timed region, every step
    cpu_baseline   oracle C restatement of the reference's one-scan-per-constraint DataFusion schedule,
               all host cores, on a bounded row sample (rank 0, N=1 only)
    --impl reference   times that CPU restatement alone (the reference itself is Rust + DataFusion and
               cannot be built in this image: no cargo/rustc; see DESIGN.md)
    --dump-outputs DIR   after the timed steps, writes the suite's results of the last step (rank 0) as
               DIR/metric.npy and DIR/status.npy (float64, one entry per constraint in suite order), so that two
               builds run with the same arguments (hence the same seeded inputs) can be compared output for output
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ROWS_PER_GPU = int(os.environ.get("TG_BENCH_ROWS", 100_000_000))
NULL_FRACTION = 0.05
METRIC = "rows/sec scanned per suite (numeric business-rules suite, 100M rows x 8 cols per GPU)"
UNIT = "rows/s"
SUITE_COLUMNS = ("f0", "f1", "f2", "i0")  # columns the literal suite references


def algorithmic_bytes(n_rows, columns=SUITE_COLUMNS):
    """SURVEY §8d: 8 B value + 1/8 B validity per referenced, nullable column, each counted once."""
    return len(columns) * (n_rows * 8 + (n_rows + 7) // 8)


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(n_rows):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE scan_kernel launch from the committed ncu --set full capture
    (profiles/scan_traffic.json), scaled by rows when the bench runs at another size; None if the file is absent."""
    p = os.path.join(ROOT, "profiles", "scan_traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        t = json.load(f)
    return int((t["dram_bytes_read"] + t["dram_bytes_write"]) * (n_rows / t["rows"]))


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region. The region is tens of milliseconds, far
    shorter than an `nvidia-smi -lms` period, so the sampler polls NVML directly (nvidia_ml_py) from a thread
    every ~1 ms; `nvidia-smi` (the B200_PROFILING.md recipe's query) is the fallback when NVML cannot be loaded."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []
        self.nvml, self.handle, self.samples, self.stop_flag = None, None, [], False
        self.smax = None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.gpu])
            except (ValueError, IndexError):
                pass
        return self.gpu

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self._physical_index()), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                reasons = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                self.samples.append((sm, reasons))
            except Exception:
                break
            time.sleep(0.001)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=2)
            n = self.nvml
            bits = {"hw_slowdown": n.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": n.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksEventReasonSwPowerCap}
            sm = [s for s, _ in self.samples]
            reasons = sorted(nm for nm, b in bits.items() if any(r & b for _, r in self.samples))
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.smax, "samples": len(sm),
                    "reasons": reasons, "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------ data ----
HOST_BLOCK_ROWS = 10_000_000  # seeded block the host table is tiled from (a multiple of 8: bitmaps tile bytewise)
HOST_SEED = 1234


def make_host_table(rows, seed=HOST_SEED, pinned=False):
    """THE table of the C2 workload — the suite's four referenced columns as host Arrow buffers (values + LSB-first
    validity bitmaps, 5 % NULLs), `rows` rows: one seeded numpy block of HOST_BLOCK_ROWS rows tiled to length (numpy's
    generators are single-threaded; a scan does not care that the block repeats). BOTH arms consume these bytes: the
    GPU arm copies them to HBM (resident leg) / stages them every step (e2e leg), the CPU arm scans them in place.
    Returns {name: (values ndarray, bitmap ndarray)}; with pinned=True the arrays are views of pinned torch tensors
    (kept alive in the returned dict under '_keep')."""
    import numpy as np
    blk = min(rows, HOST_BLOCK_ROWS)
    reps = (rows + blk - 1) // blk
    rng = np.random.default_rng(seed)
    f0 = rng.normal(100.0, 15.0, blk)
    f1 = 0.8 * f0 + rng.normal(0.0, 9.0, blk)
    f2 = rng.uniform(0.0, 1000.0, blk)
    i0 = rng.integers(-10**6, 10**6 + 1, blk)
    out, keep = {}, []
    if pinned:
        import torch
    for name, vals in (("f0", f0), ("f1", f1), ("f2", f2), ("i0", i0)):
        valid = rng.random(blk) >= NULL_FRACTION
        bm_bytes = (rows + 7) // 8
        bm_len = bm_bytes + (-bm_bytes) % 64 + 64
        if pinned:
            tv = torch.empty(rows + 64, dtype=torch.float64 if vals.dtype == np.float64 else torch.int64).pin_memory()
            tb = torch.zeros(bm_len, dtype=torch.uint8).pin_memory()
            keep += [tv, tb]
            v, bm = tv.numpy(), tb.numpy()
            v[rows:] = 0
        else:
            v, bm = np.empty(rows, dtype=vals.dtype), np.zeros(bm_len, dtype=np.uint8)
        if reps > 1 and blk % 8 == 0:
            bits = np.packbits(valid.astype(np.uint8), bitorder="little")
            for r in range(reps):
                lo, hi = r * blk, min(rows, (r + 1) * blk)
                v[lo:hi] = vals[: hi - lo]
                bm[lo // 8: lo // 8 + (hi - lo + 7) // 8] = bits[: (hi - lo + 7) // 8]
            if rows % 8:
                bm[rows // 8] &= (1 << (rows % 8)) - 1
        else:
            full = np.tile(valid, reps)[:rows]
            v[:rows] = np.tile(vals, reps)[:rows]
            packed = np.packbits(full.astype(np.uint8), bitorder="little")
            bm[: len(packed)] = packed
        out[name] = (v[:rows], bm)
    out["_keep"] = keep
    return out


def make_filler_columns(torch, n, seed, device):
    """the four columns of the 100 M x 8 table the literal suite does not reference (f3, i1..i3), generated on the device"""
    from term_b200 import _ffi as F
    from tools.bench_suites import validity
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    cols, keep = {}, []
    f3 = torch.zeros(n + 64, dtype=torch.float64, device=device)
    f3[:n].normal_(0.0, 1.0, generator=g).exp_()
    v = validity(n, g, device, NULL_FRACTION)
    cols["f3"] = dict(dtype=F.TG_FLOAT64, n_rows=n, values=f3.data_ptr(), validity=v.data_ptr())
    keep += [f3, v]
    for k in range(1, 4):
        t = torch.zeros(n + 64, dtype=torch.int64, device=device)
        t[:n].random_(-10**6, 10**6 + 1, generator=g)
        v = validity(n, g, device, NULL_FRACTION)
        cols[f"i{k}"] = dict(dtype=F.TG_INT64, n_rows=n, values=t.data_ptr(), validity=v.data_ptr())
        keep += [t, v]
    return cols, keep


def make_device_table(torch, n, seed, device):
    """(used by tests/test_gpu_full_size.py; the bench itself feeds both arms from make_host_table) Synthetic C2 table generated on the device: f0..f3 f64, i0..i3 i64, 5 % nulls, f1 = 0.8 f0 + noise.
    Buffers carry 64 elements of slack so TMA tiles may over-read the tail."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    cols, keep = {}, []
    pad = 64

    def buf(dtype):
        t = torch.zeros(n + pad, dtype=dtype, device=device)
        keep.append(t)
        return t

    def validity():
        words = (n + 63) // 64 * 8 + 64
        bits = torch.zeros(words, dtype=torch.uint8, device=device)
        chunk = 1 << 26
        w = torch.tensor([1, 2, 4, 8, 16, 32, 64, 128], dtype=torch.uint8, device=device)
        for s in range(0, n, chunk):
            e = min(n, s + chunk)
            m = (torch.rand(e - s, generator=g, device=device) >= NULL_FRACTION)
            padn = (-(e - s)) % 8
            if padn:
                m = torch.cat([m, torch.zeros(padn, dtype=torch.bool, device=device)])
            packed = (m.view(-1, 8).to(torch.uint8) * w).sum(dim=1, dtype=torch.int32).to(torch.uint8)
            bits[s // 8: s // 8 + packed.numel()] = packed
        keep.append(bits)
        return bits

    f0 = buf(torch.float64)
    f0[:n].normal_(100.0, 15.0, generator=g)
    f1 = buf(torch.float64)
    f1[:n].normal_(0.0, 9.0, generator=g)
    f1[:n].add_(f0[:n], alpha=0.8)
    f2 = buf(torch.float64)
    f2[:n].uniform_(0.0, 1000.0, generator=g)
    f3 = buf(torch.float64)
    f3[:n].normal_(0.0, 1.0, generator=g).exp_()
    floats = {"f0": f0, "f1": f1, "f2": f2, "f3": f3}
    ints = {}
    for k in range(4):
        t = buf(torch.int64)
        t[:n].random_(-10**6, 10**6 + 1, generator=g)
        ints[f"i{k}"] = t
    from term_b200 import _ffi as F
    for name, t in list(floats.items()) + list(ints.items()):
        v = validity()
        cols[name] = dict(dtype=F.TG_FLOAT64 if name[0] == "f" else F.TG_INT64, n_rows=n, values=t.data_ptr(),
                          validity=v.data_ptr(), tensor=t, bits=v)
    return cols, keep


def build_suite(T, table_name):
    A = T.Assertion
    check = (T.Check.builder("business_rules")
             .has_size(A.GreaterThan(0.0))
             .has_min("f0", A.GreaterThan(-1000.0))
             .has_mean("f1", A.Between(50.0, 110.0))
             .has_correlation("f0", "f1", A.GreaterThan(0.5))
             .satisfies("f2 > 0 AND i0 < 1000000")
             .build())
    return T.ValidationSuite.builder("numeric_business_rules").table_name(table_name).check(check).build()


def build_full_suite(T, table_name):
    """'full numeric set' variant of SURVEY §8d: {completeness,min,max,mean,sum,stddev} x 8 cols + 4 pairs"""
    A = T.Assertion
    cb = T.Check.builder("full_numeric_set").has_size(A.GreaterThan(0.0))
    names = [f"f{k}" for k in range(4)] + [f"i{k}" for k in range(4)]
    for c in names:
        cb.completeness(c, 0.9)
        for s in ("Min", "Max", "Mean", "Sum", "StandardDeviation"):
            cb.statistic(c, T.StatisticType[s], A.GreaterThan(-1e300))
    for a, b in (("f0", "f1"), ("f2", "f3"), ("i0", "i1"), ("f0", "i2")):
        cb.has_correlation(a, b, A.GreaterThan(-2.0))
    return T.ValidationSuite.builder("full_numeric_set").table_name(table_name).check(cb.build()).build()


WORKLOAD = ("C2 numeric business-rules suite (has_size, has_min(f0), has_mean(f1), has_correlation(f0,f1), "
            "satisfies(f2 > 0 AND i0 < 1000000)) on 100M rows x 8 f64/i64 cols, 5% nulls, per GPU")


def bench_config(world):
    """the `config` object of the JSON line — identical keys and workload text in both arms"""
    return {"workload": WORKLOAD, "rows_per_gpu": ROWS_PER_GPU, "columns": 8, "referenced_columns": list(SUITE_COLUMNS),
            "null_fraction": NULL_FRACTION, "parallelism": f"row-partitioned x{world}",
            "host_table": f"numpy seed {HOST_SEED} + rank, {HOST_BLOCK_ROWS}-row block tiled: the same bytes feed the GPU arm and the CPU arm"}


# ------------------------------------------------------------------------------ CPU arm ----
def _cpu_metrics(m):
    return [{"name": "size", "metric": m["size"]}, {"name": "min", "metric": m["min_f0"]}, {"name": "mean", "metric": m["mean_f1"]},
            {"name": "correlation", "metric": m["corr_f0_f1"]}, {"name": "custom_sql", "metric": m["satisfies"]}]


def time_cpu(fn, cols, rows, steps, warmup):
    for _ in range(max(1, warmup)):
        out = fn(cols, rows)
    t0 = time.perf_counter()
    for _ in range(steps):
        out = fn(cols, rows)
    dt = time.perf_counter() - t0
    return rows * steps / dt, dt / steps * 1e3, out


def pyarrow_cross_timing(cols, rows):
    """BASELINE.md §2.2: the same aggregates through pyarrow.compute (Arrow's own C++ kernels, one pass per
    aggregate, its default thread pool) on zero-copy views of the same buffers; a cross-timing, not the baseline"""
    try:
        import pyarrow as pa
        import pyarrow.compute as pc
        arr = {}
        for name in SUITE_COLUMNS:
            v, bm = cols[name]
            typ = pa.float64() if name[0] == "f" else pa.int64()
            arr[name] = pa.Array.from_buffers(typ, rows, [pa.py_buffer(bm), pa.py_buffer(v)])

        def run():
            mn = pc.min(arr["f0"]).as_py()
            mean = pc.mean(arr["f1"]).as_py()
            both = pc.and_(arr["f0"].is_valid(), arr["f1"].is_valid())
            x, y = pc.filter(arr["f0"], both), pc.filter(arr["f1"], both)
            mx, my = pc.mean(x).as_py(), pc.mean(y).as_py()
            dx, dy = pc.subtract(x, mx), pc.subtract(y, my)
            corr = pc.sum(pc.multiply(dx, dy)).as_py() / (pc.sum(pc.multiply(dx, dx)).as_py() * pc.sum(pc.multiply(dy, dy)).as_py()) ** 0.5
            sat = pc.sum(pc.and_kleene(pc.greater(arr["f2"], 0.0), pc.less(arr["i0"], 1000000)).cast(pa.int64())).as_py() / rows
            return {"size": float(rows), "min_f0": mn, "mean_f1": mean, "corr_f0_f1": corr, "satisfies": sat}
        run()
        t0 = time.perf_counter()
        out = run()
        dt = time.perf_counter() - t0
        return {"value": rows / dt, "unit": UNIT, "ms_per_step": dt * 1e3, "threads": pa.cpu_count(), "results": _cpu_metrics(out)}
    except Exception as ex:  # a cross-timing must never fail the bench
        return {"unavailable": str(ex)[:200]}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rows = int(os.environ.get("TG_BENCH_CPU_ROWS", ROWS_PER_GPU))
    from oracle import cpu_scan as S
    cores = S.use_all_host_threads()  # under torchrun every rank inherits OMP_NUM_THREADS=1
    cols = make_host_table(rows, HOST_SEED)
    value, ms, out = time_cpu(S.numeric_suite, cols, rows, args.steps, args.warmup)
    fused_value, fused_ms, fused_out = time_cpu(S.numeric_suite_fused, cols, rows, max(1, args.steps // 2), 1)
    sample_desc = (f"{rows} rows x 4 referenced cols per step ({'the full' if rows == ROWS_PER_GPU else 'a sample of the'} "
                   f"100M-row workload of one GPU; the table of rank 0 of the GPU arm, byte for byte), one full scan per constraint as "
                   f"ValidationSuite::run_sequential does, CORR in one pass like DataFusion's accumulator, OpenMP over {cores} host threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": bench_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample_desc},
        "cpu_baseline_fused": {"value": fused_value, "unit": UNIT, "cores": cores, "kind": "port", "ms_per_step": fused_ms,
                               "sample": "same rows, the whole suite in ONE scan (oracle/cpu_scan.c to_fused_c2): what the reference's "
                                         "optimizer/ would do if ValidationSuite::run invoked it (BASELINE.md §2.2)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "results": _cpu_metrics(out), "results_fused": _cpu_metrics(fused_out),
        "note": "CPU restatement of the reference's DataFusion path (oracle/cpu_scan.c); the Rust reference cannot be built in this image",
    }
    print(json.dumps(line), flush=True)


def check_gpu_against_cpu(gpu_results, cpu):
    """both arms ran on the same bytes: min / predicate ratio / size bit-exact, mean 1e-9, correlation 1e-6 (BASELINE.json)"""
    got = {r.name: r.metric for r in gpu_results}
    assert got["size"] == cpu["size"], (got, cpu)
    assert got["min"] == cpu["min_f0"], (got["min"], cpu["min_f0"])
    assert got["custom_sql"] == cpu["satisfies"], (got["custom_sql"], cpu["satisfies"])
    assert abs(got["mean"] - cpu["mean_f1"]) <= 1e-9 * abs(cpu["mean_f1"]), (got["mean"], cpu["mean_f1"])
    assert abs(got["correlation"] - cpu["corr_f0_f1"]) <= 1e-6, (got["correlation"], cpu["corr_f0_f1"])
    return "GPU results equal the CPU arm's on the same host table (size / min / predicate ratio exact, mean 1e-9, correlation 1e-6)"


def dump_outputs(results, out_dir):
    """the ConstraintResults a caller of the timed plan receives, as arrays: metric (NaN when a result has none) and
    status (ConstraintStatus value: 0 Success, 1 Failure, 2 Skipped), in suite order"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "metric.npy"), np.array([np.nan if r.metric is None else r.metric for r in results], dtype=np.float64))
    np.save(os.path.join(out_dir, "status.npy"), np.array([r.status.value for r in results], dtype=np.float64))


# ------------------------------------------------------------------------------ GPU arm ----
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="termgpu")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--variants", action="store_true", help="(kept for old scripts: the full numeric set is one of the suites now)")
    ap.add_argument("--suites", default="all", help="'all', 'none' or a comma list of c1,c2full,c3,c4,c5,mixed")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/metric.npy and DIR/status.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; it does not apply to --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    import term_b200 as T
    from term_b200 import _ffi as F
    from term_b200.distributed import bind_to_gpu_numa, execute_distributed
    from tools import bench_suites as BS

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    # N > 1: every rank stages host buffers at once; keep each rank's pinned memory on its GPU's socket. N = 1 keeps
    # all host cores (the cpu_baseline leg uses them)
    numa_cpus = bind_to_gpu_numa(local_rank) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    n = ROWS_PER_GPU
    ctx = T.SessionContext(local_rank)
    # the host table (pinned): rank r's shard is the seeded table HOST_SEED + r; rank 0's is the CPU arm's table
    host = make_host_table(n, HOST_SEED + rank, pinned=True)
    keep, cols = [], {}
    for name in SUITE_COLUMNS:
        v, bm = host[name]
        tv = torch.zeros(n + 64, dtype=torch.float64 if name[0] == "f" else torch.int64, device=device)
        tv[:n].copy_(torch.from_numpy(v), non_blocking=True)
        tb = torch.from_numpy(bm).to(device, non_blocking=True)
        keep += [tv, tb]
        cols[name] = dict(dtype=F.TG_FLOAT64 if name[0] == "f" else F.TG_INT64, n_rows=n, values=tv.data_ptr(), validity=tb.data_ptr())
    fill, fkeep = make_filler_columns(torch, n, 42 + 2 + rank, device)
    cols.update(fill)
    keep += fkeep
    torch.cuda.synchronize()
    ctx.register_device_table("data", cols, keepalive=keep)

    suite = build_suite(T, "data")
    plan, slots = suite.build_plan()
    engine_stream = torch.cuda.ExternalStream(ctx.stream(), device=device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        if world > 1:
            execute_distributed(plan, ctx, "data")
        else:
            plan.execute(ctx, "data")

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count()
    scan_ms = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(engine_stream)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
        scan_ms.append(plan.stats()["scan_ms"])
    ev1.record(engine_stream)
    barrier()
    wall = time.perf_counter() - t0
    dev_ms = ev0.elapsed_time(ev1)
    launches = ctx.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    # max over ranks of the device-side time
    t_ms = torch.tensor([dev_ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    total_ms = float(t_ms.item())
    ms_per_step = total_ms / args.steps
    value = n * world * args.steps / (total_ms / 1e3)

    results = [plan.result(s) for _, _, s in slots]
    if args.dump_outputs and rank == 0:
        dump_outputs(results, args.dump_outputs)
    kernel_ms = sum(scan_ms) / len(scan_ms)
    alg_bytes = algorithmic_bytes(n)
    peak, peak_src = measured_peak_gbs()
    achieved = alg_bytes / (kernel_ms / 1e3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": measured_traffic(n), "kernel": "scan_kernel (+ scan_finalize_kernel)", "kernel_ms": kernel_ms,
                "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                "step_gbs": alg_bytes * world / (ms_per_step / 1e3) / 1e9}

    # ---------------- e2e: host Arrow buffers -> H2D -> scan -> results, every step ----------------
    e2e = None
    if not args.no_e2e:
        e2e_rows = int(os.environ.get("TG_BENCH_E2E_ROWS", n))
        h2d_bytes = sum(e2e_rows * 8 + (e2e_rows + 7) // 8 for _ in SUITE_COLUMNS)
        esuite = build_suite(T, "e2e")
        eplan, eslots = esuite.build_plan()

        def e2e_step():
            t = ctx._create("e2e")
            for name in SUITE_COLUMNS:
                v, bm = host[name]
                dt = F.TG_FLOAT64 if name[0] == "f" else F.TG_INT64
                F.check(F.lib().tg_table_append_host(t, name.encode(), dt, e2e_rows, v.ctypes.data, None, bm.ctypes.data, 0))
            if world > 1:
                execute_distributed(eplan, ctx, "e2e")
            else:
                eplan.execute(ctx, "e2e")
            out = [eplan.result(s) for _, _, s in eslots]
            ctx.deregister_table("e2e")
            return out

        e2e_steps = max(3, min(args.steps, 5))
        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            eres = e2e_step()
        barrier()
        e2e_wall = time.perf_counter() - t0
        tw = torch.tensor([e2e_wall], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        e2e_value = e2e_rows * world * e2e_steps / float(tw.item())
        d2h = 5 * 8 + 64  # one ScanAggOut record per aggregate + 5 result structs
        e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h * 4,
               "steps": e2e_steps, "rows_per_step_per_gpu": e2e_rows, "ms_per_step": float(tw.item()) / e2e_steps * 1e3,
               "note": "pinned host Arrow buffers -> tg_table_append_host (async H2D) -> tg_plan_execute -> tg_plan_result; at N = 1 "
                       "this is the PCIe link (3.25 GB per step), not the engine"}
        if e2e_rows == n:
            assert [(r.status, r.metric) for r in eres] == [(r.status, r.metric) for r in results], "e2e and resident results differ"

    cpu_baseline = cpu_fused = pyarrow_x = parity = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import cpu_scan as S
        cores = S.use_all_host_threads()
        sample = int(os.environ.get("TG_BENCH_CPU_ROWS", n))
        hcols = {k: (v[0][:sample], v[1]) for k, v in host.items() if k != "_keep"}
        rate, ms, out = time_cpu(S.numeric_suite, hcols, sample, 20, 1)
        frate, fms, fout = time_cpu(S.numeric_suite_fused, hcols, sample, 10, 1)
        what = "the full per-GPU workload (the very table the GPU arm scanned)" if sample == n else "a prefix of the GPU arm's table"
        cpu_baseline = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "ms_per_step": ms,
                        "sample": f"{sample} rows: {what}, 20 repeats after warm-up; oracle/cpu_scan.c: one full scan per constraint "
                                  f"(run_sequential schedule), CORR in one pass, OpenMP over {cores} host threads",
                        "results": _cpu_metrics(out)}
        cpu_fused = {"value": frate, "unit": UNIT, "cores": cores, "kind": "port", "ms_per_step": fms,
                     "sample": f"{sample} rows, the whole suite in ONE scan (to_fused_c2), 10 repeats", "results": _cpu_metrics(fout)}
        pyarrow_x = pyarrow_cross_timing(hcols, sample)
        if sample == n:
            parity = check_gpu_against_cpu(results, out)
            check_gpu_against_cpu(results, fout)

    # ---------------- the other configs: one line each in `suites` ----------------
    suites = []
    if args.suites != "none":
        which = ["c1", "c2full", "c3", "c4", "c5", "mixed"] if args.suites == "all" else args.suites.split(",")
        suites = BS.run_driver_suites(which, ctx, device, world, rank, peak, steps=int(os.environ.get("TG_BENCH_SUITE_STEPS", 5)),
                                      c2_table="data", build_full_suite=build_full_suite)

    if rank == 0:
        cfg = bench_config(world)
        cfg.update({"l2": "inputs (3.25 GB/step) are larger than L2; no flush needed",
                    "merge": ("fixed-size partial aggregates exchanged through peer mailboxes (P2P stores over NVLink, "
                              "tg_plan_exchange_and_finalize); NCCL all-gather for variable-size partials") if world > 1 else "single GPU",
                    "numa_bound_cpus": len(numa_cpus) if numa_cpus else 0})
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": cfg,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "cpu_baseline_fused": cpu_fused, "pyarrow_cross_timing": pyarrow_x,
            "parity_vs_cpu_arm": parity, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clocks, "wall_ms_per_step": wall / args.steps * 1e3,
            "results": [{"name": r.name, "status": r.status.name, "metric": r.metric} for r in results],
            "suites": suites,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
