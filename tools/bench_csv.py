r"""Registration of a CSV file (csv.cu: the K8a tokenizer and the K8b column parsers).

File, written into a temporary directory from a seeded generator: --rows records of Int64, Float64 (repr), Boolean, Utf8
(C3-shaped emails, 10 % quoted with a comma inside, 2 % empty = NULL), Date32 and Timestamp(Microsecond) columns, several GB
at the default size. Timed, each over --steps runs after one warm-up (host clock, ending in a device synchronise):
  register_csv                  the GPU path
  pyarrow.csv.read_csv + register_table   the host path (pyarrow's reader on all threads, then the Arrow copy)
  register_parquet              the same data written as Parquet (Snappy)
Also: the bytes copied host to device (the file's bytes: every window crosses PCIe once), the bytes copied device to device
(the record a chunk edge cuts off is moved in front of the next window; computed here from the file, which has no quoted
line breaks), and in a separate profiled run (torch.profiler, CUDA activities: the device's start / end timestamps of every
kernel, no host clock) the device time of each CSV kernel. One JSON line on stdout
(and in --out when given), with the card's name and power limit read in the same process.

    python tools/bench_csv.py [--rows 40000000] [--steps 3] [--out FILE] [--dialect dump] [--csv-only]

--dialect dump writes the file as a database dump: the quoted emails carry a \" escape, NULL emails are \N and every block
of 1 M records follows a # comment line; it is registered with escape '\', comment '#' and null_regex ^\\N$. pyarrow's
reader has no comment lines, so that dialect times register_csv only, as --csv-only does for either.
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
import pyarrow.csv as pacsv
import pyarrow.parquet as pq

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

KERNELS = ("csv_tok_pass1_kernel", "csv_tok_scan_kernel", "csv_tok_pass2_kernel", "csv_tok_finish_kernel", "csv_parse_kernel",
           "csv_tail_kernel", "merge_bits_kernel", "pq_block_scan_kernel", "pq_str_write_kernel")

SCHEMA = pa.schema([pa.field("id", pa.int64()), pa.field("x", pa.float64()), pa.field("flag", pa.bool_()), pa.field("email", pa.string()),
                    pa.field("day", pa.date32()), pa.field("ts", pa.timestamp("us"))])


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, limit = [x.strip() for x in q.stdout.strip().split(",")[:2]] if q.returncode == 0 and q.stdout.strip() else ("unknown", "unknown")
    return {"gpu": name, "power_limit": limit}


DUMP = dict(escape="\\", comment="#", null_regex=r"^\\N$")


def write_csv(path, n, seed, dump=False):
    rng = np.random.default_rng(seed)
    step = 1_000_000
    with open(path, "w") as f:
        f.write(",".join(SCHEMA.names) + "\n")
        for lo in range(0, n, step):
            if dump:
                f.write(f'# block {lo},"x\n')
            idx = np.arange(lo, min(n, lo + step))
            m = len(idx)
            ids = rng.integers(-10**15, 10**15, m).astype(str)
            xs = np.array([repr(v) for v in rng.normal(100.0, 15.0, m).tolist()])
            flag = np.where(rng.random(m) < 0.5, "true", "false")
            em = np.char.add(np.char.add("user", idx.astype(str)), "@example.com")
            em = np.where(idx % 10 == 0, np.char.add(np.char.add('"\\"' if dump else '"', np.char.replace(em, "@", ",x@")), '"'), em)
            em = np.where(idx % 50 == 7, "\\N" if dump else "", em)
            days = rng.integers(-20000, 30000, m)
            day = np.datetime_as_string(days.astype("datetime64[D]"))
            ts = np.datetime_as_string((days * 86_400_000_000 + rng.integers(0, 86_400_000_000, m)).astype("datetime64[us]"))
            cols = [ids, xs, flag, em, day, ts]
            line = cols[0]
            for c in cols[1:]:
                line = np.char.add(np.char.add(line, ","), c)
            f.write("\n".join(line.tolist()) + "\n")


def carry_bytes(path, window):
    """bytes the chunk pipeline copies device to device: at every window edge, the part of the chunk after its last complete
    record (the file has no quoted line breaks, so that is the part after the last LF)"""
    import mmap
    total, start = 0, 0
    with open(path, "rb") as f, mmap.mmap(f.fileno(), 0, prot=mmap.PROT_READ) as mm:
        size = len(mm)
        for edge in range(window, size, window):
            p = mm.rfind(b"\n", start, edge)
            carry = edge - start if p < 0 else edge - (p + 1)
            total += carry
            start = edge - carry
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=40_000_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--dialect", choices=["default", "dump"], default="default")
    ap.add_argument("--csv-only", action="store_true")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    import torch
    import term_b200 as T
    if not torch.cuda.is_available():
        sys.exit("bench_csv.py needs a CUDA device")
    torch.cuda.set_device(0)
    tmp = tempfile.mkdtemp(prefix="tg_bench_csv_")
    path = os.path.join(tmp, "data.csv")
    dump = a.dialect == "dump"
    csv_only = a.csv_only or dump
    opts = DUMP if dump else {}
    write_csv(path, a.rows, 1, dump)
    ro = pacsv.ReadOptions(column_names=SCHEMA.names, skip_rows=1)
    po = pacsv.ParseOptions(newlines_in_values=True)
    co = pacsv.ConvertOptions(column_types=SCHEMA, strings_can_be_null=True, quoted_strings_can_be_null=True, null_values=[""],
                              true_values=["true"], false_values=["false"])
    pq_path = os.path.join(tmp, "data.parquet")
    if not csv_only:
        pq.write_table(pacsv.read_csv(path, read_options=ro, parse_options=po, convert_options=co), pq_path, compression="SNAPPY")
    ctx = T.SessionContext(0)

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

    csv_ms, csv_runs = timed(lambda: ctx.register_csv("bench", path, SCHEMA, **opts))
    arrow_ms = arrow_runs = pq_ms = pq_runs = None
    if not csv_only:
        arrow_ms, arrow_runs = timed(lambda: ctx.register_table("bench", pacsv.read_csv(path, read_options=ro, parse_options=po, convert_options=co)))
        pq_ms, pq_runs = timed(lambda: ctx.register_parquet("bench", pq_path))
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        ctx.register_csv("bench", path, SCHEMA, **opts)
        ctx.sync_copies()
        torch.cuda.synchronize()
    ctx.deregister_table("bench")
    kern = {}
    for ev in prof.key_averages():
        for k in KERNELS:
            if k in ev.key:
                kern[k] = kern.get(k, 0.0) + ev.device_time_total / 1e3
    size = os.path.getsize(path)
    window = int(os.environ.get("TG_CSV_CHUNK_BYTES") or 0) or 256 << 20  # as csv.cu reads it
    rec = {"workload": f"register one CSV file of {a.rows} records x 6 columns (Int64, Float64, Boolean, Utf8 with quoting, Date32, Timestamp(us))",
           "dialect": a.dialect,
           "rows": a.rows, "file_bytes": size, "steps": a.steps,
           "timing": "host clock around the registration + device synchronise; mean of the timed runs after one warm-up",
           "kernel_timing": "torch.profiler CUDA activities, one registration in a separate run", **card(),
           "register_csv_ms": csv_ms, "register_csv_ms_runs": csv_runs, "h2d_bytes": size, "h2d_gbs": round(size / (csv_ms / 1e3) / 1e9, 2),
           "chunk_bytes": window, "d2d_carry_bytes": carry_bytes(path, window),
           "pyarrow_read_csv_plus_register_table_ms": arrow_ms, "pyarrow_runs": arrow_runs,
           "register_parquet_ms": pq_ms, "register_parquet_runs": pq_runs, "parquet_bytes": None if csv_only else os.path.getsize(pq_path),
           "kernel_ms": {k: round(v, 3) for k, v in kern.items()}, "kernel_ms_total": round(sum(kern.values()), 3)}
    ctx.close()
    os.remove(path)
    if not csv_only:
        os.remove(pq_path)
    os.rmdir(tmp)
    out = json.dumps(rec)
    print(out, flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
