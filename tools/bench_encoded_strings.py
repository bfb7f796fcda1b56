"""Registration of a C3-shaped string column (25 M rows, lengths ~ Poisson(24) clipped to [8, 64], 2 % NULL) from host Arrow
arrays: plain Utf8 against dictionary<int16 | int32, utf8> at 1 000 and 1 M distinct values and utf8_view. The encoded forms
are decoded to Utf8 on the device (tables.cu: arrow_dict_locate_kernel / arrow_view_locate_kernel, then the shared
pq_block_scan_kernel / pq_str_write_kernel); what crosses PCIe is the encoded form.

Per configuration: the wall time of register_table (host clock, ending in a device synchronise) over --steps timed runs
after one warm-up, the bytes the engine copies host -> device, and in a separate profiled run (torch.profiler, CUDA
activities) the device time of each decode kernel. One JSON line on stdout (and in --out when given), with the card's name
and power limit read in the same process.

    python tools/bench_encoded_strings.py [--rows 25000000] [--steps 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

KERNELS = ("arrow_dict_locate_kernel", "arrow_view_locate_kernel", "pq_block_scan_kernel", "pq_str_write_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, limit = [x.strip() for x in q.stdout.strip().split(",")[:2]] if q.returncode == 0 and q.stdout.strip() else ("unknown", "unknown")
    return {"gpu": name, "power_limit": limit}


def vocab(k, rng):
    """k distinct C3-shaped strings: 70 % e-mail shaped, 10 % SSN shaped, the rest free text"""
    lens = np.clip(rng.poisson(24, k), 8, 64)
    out = []
    for i in range(k):
        if i % 10 < 7:
            s = f"u{i}@ex{i % 97}.com"
        elif i % 10 == 7:
            s = f"{100 + i % 800:03d}-{10 + i % 89:02d}-{i % 10000:04d}|{i}"
        else:
            s = f"text {i} "
        out.append(s + "x" * max(0, int(lens[i]) - len(s)))
    return out


def column(n, k, seed):
    rng = np.random.default_rng(seed)
    codes = rng.integers(0, k, n).astype(np.int32)
    valid = rng.random(n) >= 0.02
    return pa.DictionaryArray.from_arrays(pa.array(codes, mask=~valid), pa.array(vocab(k, rng), type=pa.string()))


def h2d_bytes(arr):
    """bytes the engine copies host -> device for one column (engine bookkeeping of a few bytes per 1024 rows included)"""
    n = len(arr)
    bits = (n + 7) // 8 if arr.null_count else 0
    blocks = 24 * ((n + 1023) // 1024)
    t = arr.type
    if pa.types.is_dictionary(t):
        d = arr.dictionary
        do = np.frombuffer(d.buffers()[1], dtype=np.int32 if pa.types.is_string(d.type) else np.int64)
        return n * t.index_type.bit_width // 8 + int(do[d.offset + len(d)] - do[d.offset]) + 8 * len(d) + bits + blocks
    if t == pa.string_view():
        data = sum(b.size for b in arr.buffers()[2:] if b is not None)
        return 16 * n + data + bits + blocks + 16 * (len(arr.buffers()) - 2)
    offs = np.frombuffer(arr.buffers()[1], dtype=np.int32)
    return 4 * (n + 1) + int(offs[arr.offset + n] - offs[arr.offset]) + bits


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=25_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    import torch
    import term_b200 as T
    if not torch.cuda.is_available():
        sys.exit("bench_encoded_strings.py needs a CUDA device")
    torch.cuda.set_device(0)
    ctx = T.SessionContext(0)
    n = a.rows
    d1k, d1m = column(n, 1000, 1), column(n, 1_000_000, 2)
    configs = [("utf8_1k", pc.cast(d1k, pa.string())),
               ("dict_int16_1k", pa.DictionaryArray.from_arrays(d1k.indices.cast(pa.int16()), d1k.dictionary)),
               ("dict_int32_1k", d1k),
               ("utf8_1m", pc.cast(d1m, pa.string())),
               ("dict_int32_1m", d1m),
               ("view_1k", pc.cast(pc.cast(d1k, pa.string()), pa.string_view()))]
    lines = {"workload": "register a C3-shaped string column from host Arrow (25 M rows, avg 24 B, 2 % NULL)", "rows": n, "steps": a.steps,
             "timing": "host clock around register_table + device synchronise; mean of the timed runs after one warm-up",
             "kernel_timing": "torch.profiler CUDA activities, one registration in a separate run", **card(),
             "not_run": {"dict_int16_1m": "Int16 indices cannot address 1 M dictionary values"}, "configs": {}}
    for name, arr in configs:
        t = pa.table({"s": arr})
        ts = []
        for i in range(a.steps + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ctx.register_table("enc", t)
            ctx.sync_copies()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
            ctx.deregister_table("enc")
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            ctx.register_table("enc", t)
            ctx.sync_copies()
            torch.cuda.synchronize()
        bufs = ctx.column_buffers("enc", "s")
        ctx.deregister_table("enc")
        kern = {}
        for ev in prof.key_averages():
            for k in KERNELS:
                if k in ev.key:
                    kern[k] = kern.get(k, 0.0) + ev.device_time_total / 1e3
        ms = sum(ts[1:]) / a.steps
        hb = h2d_bytes(arr)
        lines["configs"][name] = {"register_ms": round(ms, 3), "register_ms_runs": [round(x, 3) for x in ts[1:]], "h2d_bytes": hb,
                                  "h2d_gbs": round(hb / (ms / 1e3) / 1e9, 2), "decoded_value_bytes": int(bufs["n_value_bytes"]),
                                  "kernel_ms": {k: round(v, 4) for k, v in kern.items()}}
        print(json.dumps({name: lines["configs"][name]}), file=sys.stderr, flush=True)
    ctx.close()
    out = json.dumps(lines)
    print(out, flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
