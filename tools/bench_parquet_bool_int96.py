"""Registration of Parquet BOOLEAN and INT96 columns (parquet.cu: pq_expand_bool_kernel, pq_expand_kernel with the INT96 load).

Files, written with pyarrow (Snappy, the writer's default codec) into a temporary directory:
  bool_v1_plain   100 M-row nullable BOOLEAN column (10 % NULL), V1 data pages: PLAIN values
  bool_v2_rle     the same column, V2 data pages: RLE values
  int96_dict      25 M-row nullable INT96 column (2 % NULL, 100 000 distinct instants), dictionary-encoded: its 1.2 MB
                  dictionary outgrows the writer's 1 MiB dictionary page limit, so most pages fall back to PLAIN (the mixed
                  chunks writers produce for high-cardinality columns)
  int96_plain     25 M-row nullable INT96 column (2 % NULL, all instants distinct), PLAIN
Per file: the wall time of register_parquet (host clock, ending in a device synchronise) over --steps timed runs after one
warm-up; the same data registered from host Arrow (register_table); for the INT96 files the same instants written as an
INT64 timestamp[ns] column with the same encoding and registered with register_parquet; the bytes copied to the device
(page bodies after inflation, the validity bitmap and the block table; the run tables are not counted); and in a separate
profiled run (torch.profiler, CUDA activities) the device time of each decode kernel. One JSON line on stdout (and in
--out when given), with the card's name and power limit read in the same process.

    python tools/bench_parquet_bool_int96.py [--bool-rows 100000000] [--int96-rows 25000000] [--steps 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import pyarrow as pa
import pyarrow.parquet as pq

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

KERNELS = ("pq_expand_bool_kernel", "pq_expand_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, limit = [x.strip() for x in q.stdout.strip().split(",")[:2]] if q.returncode == 0 and q.stdout.strip() else ("unknown", "unknown")
    return {"gpu": name, "power_limit": limit}


def h2d_bytes(path):
    """page bodies (uncompressed, page headers included) + validity bitmap + 24-byte block per 1024 rows, over all chunks"""
    md = pq.ParquetFile(path).metadata
    total = 0
    for rg in range(md.num_row_groups):
        for ci in range(md.num_columns):
            cm = md.row_group(rg).column(ci)
            total += cm.total_uncompressed_size + (cm.num_values + 7) // 8 + 24 * ((cm.num_values + 1023) // 1024)
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bool-rows", type=int, default=100_000_000)
    ap.add_argument("--int96-rows", type=int, default=25_000_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    import torch
    import term_b200 as T
    if not torch.cuda.is_available():
        sys.exit("bench_parquet_bool_int96.py needs a CUDA device")
    torch.cuda.set_device(0)
    ctx = T.SessionContext(0)
    rng = np.random.default_rng(1)
    nb, nt = a.bool_rows, a.int96_rows
    b = pa.table({"v": pa.array(rng.random(nb) < 0.4, mask=rng.random(nb) < 0.10)})
    base = 1_600_000_000 * 10**9
    ts_dict = pa.table({"v": pa.array(base + rng.integers(0, 100_000, nt) * 7_919_000_003, type=pa.timestamp("ns"), mask=rng.random(nt) < 0.02)})
    ts_plain = pa.table({"v": pa.array(base + rng.permutation(nt).astype(np.int64) * 1_000_003, type=pa.timestamp("ns"), mask=rng.random(nt) < 0.02)})
    tmp = tempfile.mkdtemp(prefix="tg_bench_pq_")
    files = {}  # name -> (path, host table, INT64 twin path | None)

    def write(name, t, int96, **kw):
        p = os.path.join(tmp, name + ".parquet")
        pq.write_table(t, p, compression="SNAPPY", use_deprecated_int96_timestamps=int96, **kw)
        return p
    files["bool_v1_plain"] = (write("bool_v1_plain", b, False, data_page_version="1.0"), b, None)
    files["bool_v2_rle"] = (write("bool_v2_rle", b, False, data_page_version="2.0"), b, None)
    files["int96_dict"] = (write("int96_dict", ts_dict, True), ts_dict, write("int64_dict", ts_dict, False))
    files["int96_plain"] = (write("int96_plain", ts_plain, True, use_dictionary=False), ts_plain, write("int64_plain", ts_plain, False, use_dictionary=False))

    def timed(register):
        ts = []
        for _ in range(a.steps + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            register()
            ctx.sync_copies()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
            ctx.deregister_table("bench")
        return round(sum(ts[1:]) / a.steps, 3), [round(x, 3) for x in ts[1:]]

    lines = {"workload": "register one Parquet BOOLEAN (100 M rows, 10 % NULL) / INT96 (25 M rows, 2 % NULL) column, Snappy",
             "bool_rows": nb, "int96_rows": nt, "steps": a.steps,
             "timing": "host clock around register_parquet / register_table + device synchronise; mean of the timed runs after one warm-up",
             "kernel_timing": "torch.profiler CUDA activities, one registration in a separate run", **card(), "files": {}}
    for name, (path, host, twin) in files.items():
        ms, runs = timed(lambda: ctx.register_parquet("bench", path))
        arrow_ms, _ = timed(lambda: ctx.register_table("bench", host))
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            ctx.register_parquet("bench", path)
            ctx.sync_copies()
            torch.cuda.synchronize()
        ctx.deregister_table("bench")
        kern = {}
        for ev in prof.key_averages():
            for k in KERNELS:
                if k in ev.key:
                    kern[k] = kern.get(k, 0.0) + ev.device_time_total / 1e3
        hb = h2d_bytes(path)
        rec = {"register_parquet_ms": ms, "register_parquet_ms_runs": runs, "register_arrow_ms": arrow_ms, "file_bytes": os.path.getsize(path),
               "h2d_bytes": hb, "h2d_gbs": round(hb / (ms / 1e3) / 1e9, 2), "kernel_ms": {k: round(v, 4) for k, v in kern.items()}}
        if twin:
            rec["int64_timestamp_parquet_ms"], _ = timed(lambda: ctx.register_parquet("bench", twin))
        lines["files"][name] = rec
        print(json.dumps({name: rec}), file=sys.stderr, flush=True)
    ctx.close()
    for p, _, twin in files.values():
        os.remove(p)
        if twin:
            os.remove(twin)
    os.rmdir(tmp)
    out = json.dumps(lines)
    print(out, flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
