"""Registration of RecordBatches that are already in HBM, through the Arrow C Device Data Interface
(SessionContext.register_arrow_device -> tg_table_append_arrow_device), against register_table of the same batches from host
Arrow. Workloads: a C2-shaped table (100 M rows x f0..f3 Float64, i0..i3 Int64, 5 % NULL) and the C3-shaped string column
(25 M rows, ~24 B, 2 % NULL) as Utf8, as dictionary<int32, utf8> (1 000 values) and as Utf8View.

Per workload: the wall time of each registration (host clock around the call, which returns after its device work; mean of
--steps runs after one warm-up), in a separate profiled run (torch.profiler, CUDA activities) the device time of the
kernels and device-to-device copies of one device registration, the bytes that registration must read and write in HBM
and their time at the 7.7 TB/s data-sheet bandwidth, and a check that a suite gives the same results on both tables.
One JSON line on stdout (and in --out), with the card's name and power limit read in the same process.

    python tools/bench_arrow_device.py [--rows 100000000] [--string-rows 25000000] [--steps 3] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.bench_encoded_strings import card, column  # noqa: E402

HBM_PEAK = 7.7e12  # B/s, HGX B200 data sheet, one GPU


def c2_batch(n, seed=1234, blk=1 << 20):
    """f0..f3 Float64, i0..i3 Int64, 5 % NULL: one seeded block per column tiled to n rows"""
    rng = np.random.default_rng(seed)
    cols, names = [], []
    for k in range(8):
        vals = rng.normal(100.0, 15.0, blk) if k < 4 else rng.integers(-10**6, 10**6 + 1, blk)
        valid = rng.random(blk) >= 0.05
        reps = (n + blk - 1) // blk
        cols.append(pa.array(np.tile(vals, reps)[:n], mask=~np.tile(valid, reps)[:n]))
        names.append(f"f{k}" if k < 4 else f"i{k - 4}")
    return pa.record_batch(cols, names=names)


def hbm_bytes(batch):
    """bytes a device registration must read (the producer's buffers of the batch) and write (the stored columns)"""
    rd = wr = 0
    for arr in batch.columns:
        n = len(arr)
        bits = (n + 7) // 8 if arr.null_count else 0
        t = arr.type
        if pa.types.is_dictionary(t):
            d = arr.dictionary
            do = np.frombuffer(d.buffers()[1], dtype=np.int32)
            dict_b = int(do[d.offset + len(d)] - do[d.offset])
            logical = pc.cast(arr, pa.string())
            lo = np.frombuffer(logical.buffers()[1], dtype=np.int32)
            vb = int(lo[logical.offset + n] - lo[logical.offset])
            rd += n * t.index_type.bit_width // 8 + bits + dict_b
            wr += 4 * (n + 1) + vb + bits
        elif t == pa.string_view():
            data = sum(b.size for b in arr.buffers()[2:] if b is not None)
            logical = pc.cast(arr, pa.string())
            lo = np.frombuffer(logical.buffers()[1], dtype=np.int32)
            rd += 16 * n + data + bits
            wr += 4 * (n + 1) + int(lo[logical.offset + n] - lo[logical.offset]) + bits
        elif pa.types.is_string(t):
            offs = np.frombuffer(arr.buffers()[1], dtype=np.int32)
            vb = int(offs[arr.offset + n] - offs[arr.offset])
            rd += 4 * (n + 1) + vb + bits
            wr += 4 * (n + 1) + vb + bits
        else:
            rd += n * t.bit_width // 8 + bits
            wr += n * t.bit_width // 8 + bits
    return rd, wr


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--string-rows", type=int, default=25_000_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    import torch
    import term_b200 as T
    from tests.test_arrow_device import DeviceBatch, _suite
    if not torch.cuda.is_available():
        sys.exit("bench_arrow_device.py needs a CUDA device")
    torch.cuda.set_device(0)
    ctx = T.SessionContext(0)
    d1k = column(a.string_rows, 1000, 1)
    utf8 = pc.cast(d1k, pa.string())
    workloads = [("c2_100m_x8", c2_batch(a.rows), {f"f{k}": "g" for k in range(4)} | {f"i{k}": "l" for k in range(4)}),
                 ("c3_utf8", pa.record_batch([utf8], names=["s"]), {"s": "u"}),
                 ("c3_dict_int32", pa.record_batch([d1k], names=["s"]), {"s": "dict"}),
                 ("c3_utf8_view", pa.record_batch([pc.cast(utf8, pa.string_view())], names=["s"]), {"s": "vu"})]
    lines = {"workload": "register 100 M x 8 C2 columns and 25 M C3 strings from HBM-resident Arrow (device) and from host Arrow",
             "rows": a.rows, "string_rows": a.string_rows, "steps": a.steps,
             "timing": "host clock around the registration (device work included); mean of the timed runs after one warm-up",
             "kernel_timing": "torch.profiler CUDA activities (kernels + device-to-device copies), one device registration in a separate run",
             "hbm_peak_tbs": HBM_PEAK / 1e12, **card(), "configs": {}}

    def timed(fn):
        ts = []
        for _ in range(a.steps + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            ctx.sync_copies()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
            ctx.deregister_table("reg")
        return ts[1:]

    for name, batch, fmts in workloads:
        dev = DeviceBatch(batch)
        torch.cuda.synchronize()
        dev_ms = timed(lambda: ctx.register_arrow_device("reg", dev))
        host_ms = timed(lambda: ctx.register_table("reg", batch))
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            ctx.register_arrow_device("reg", dev)
            ctx.sync_copies()
            torch.cuda.synchronize()
        ctx.deregister_table("reg")
        kern, dev_total = {}, 0.0
        for ev in prof.key_averages():
            if ev.device_time_total > 0 and ev.device_type == torch.autograd.DeviceType.CUDA:
                kern[ev.key] = round(kern.get(ev.key, 0.0) + ev.device_time_total / 1e3, 4)
                dev_total += ev.device_time_total / 1e3
        ctx.register_arrow_device("reg_dev", dev)
        ctx.register_table("reg_host", batch)
        same = _suite(ctx, "reg_dev", fmts) == _suite(ctx, "reg_host", fmts)
        ctx.deregister_table("reg_dev")
        ctx.deregister_table("reg_host")
        assert same, f"{name}: the device and host registrations give different suite results"
        rd, wr = hbm_bytes(batch)
        ms = sum(dev_ms) / a.steps
        lines["configs"][name] = {"device_register_ms": round(ms, 3), "device_register_ms_runs": [round(x, 3) for x in dev_ms],
                                  "host_register_ms": round(sum(host_ms) / a.steps, 3), "host_register_ms_runs": [round(x, 3) for x in host_ms],
                                  "hbm_read_bytes": rd, "hbm_write_bytes": wr, "hbm_bound_ms": round((rd + wr) / HBM_PEAK * 1e3, 3),
                                  "device_time_ms": round(dev_total, 3), "device_time_by_name_ms": kern,
                                  "wall_share_of_hbm_bound": round((rd + wr) / HBM_PEAK * 1e3 / ms, 3), "same_suite_results": same}
        print(json.dumps({name: lines["configs"][name]}), file=sys.stderr, flush=True)
        del dev
    ctx.close()
    out = json.dumps(lines)
    print(out, flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
