#!/usr/bin/env python3
"""Cost of row verdicts (tg_plan_request_row_mask): the C3 string suite and a C2-style numeric predicate suite at their
bench sizes, each plan run with masks off and on, alternating step by step. Prints one JSON line per suite: mean GPU ms of
both arms, the extra bytes the masks write (n/8 per masked slot for the kernel words and n/8 for the exported values;
slots whose population is the column's non-null rows write a validity buffer too), and the card's name and power limit.

    python tools/bench_row_masks.py [--steps 20] [--scale 1.0] [--out row_masks.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import term_b200 as T  # noqa: E402
from term_b200 import _ffi as F  # noqa: E402
from tools.bench_suites import make_strings, validity  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def alternate(plans, ctx, table, steps):
    """plans: {arm: plan}; one warm-up each, then arms interleaved; returns {arm: (mean gpu_ms, mean wall ms)}"""
    for p in plans.values():
        p.execute(ctx, table)
    gpu = {k: [] for k in plans}
    wall = {k: [] for k in plans}
    for _ in range(steps):
        for k, p in plans.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            p.execute(ctx, table)
            wall[k].append((time.perf_counter() - t0) * 1e3)
            gpu[k].append(p.stats()["gpu_ms"])
    return {k: (sum(gpu[k]) / steps, sum(wall[k]) / steps) for k in plans}


def line(name, n, masked, res, out):
    off, on = res["off"], res["on"]
    rec = {"workload": name, "rows": n, "masked_slots": masked, "gpu_ms_off": off[0], "gpu_ms_on": on[0],
           "wall_ms_off": off[1], "wall_ms_on": on[1], "gpu_overhead": on[0] / off[0] - 1.0,
           "extra_bytes_kernel_words": masked * ((n + 31) // 32) * 4, "extra_bytes_exported": masked * ((n + 31) // 32) * 4,
           "card": card()}
    print(json.dumps(rec), flush=True)
    if out:
        with open(out, "a") as f:
            f.write(json.dumps(rec) + "\n")


def build(fn, mask):
    p = T.api.Plan()
    slots = fn(p)
    if mask:
        for s in slots:
            p.request_row_mask(s)
    return p


def c2(ctx, dev, scale, steps, out):
    """eight f64 columns (5 % NULL), one satisfies() each plus completeness: the C2 shape with row-level constraints"""
    n = int(100_000_000 * scale)
    g = torch.Generator(device=dev)
    g.manual_seed(2)
    cols, keep = {}, []
    for k in range(8):
        x = torch.randn(n, generator=g, device=dev, dtype=torch.float64) * 10 + k
        v = validity(n, g, dev, 0.05)
        keep += [x, v]
        cols[f"c{k}"] = dict(dtype=F.TG_FLOAT64, n_rows=n, values=x.data_ptr(), validity=v.data_ptr())
    ctx.register_device_table("rm_c2", cols, keepalive=keep)
    lib = F.lib()

    def slots(p):
        s = [lib.tg_plan_add_custom_sql(p.handle, f"c{k} > {k}".encode(), None) for k in range(8)]
        cs = (C.c_char_p * 1)(b"c0")
        s.append(lib.tg_plan_add_completeness(p.handle, cs, 1, 0.5, 0, 0))
        return s
    res = alternate({"off": build(slots, False), "on": build(slots, True)}, ctx, "rm_c2", steps)
    line("c2_predicates_x8_plus_completeness", n, 9, res, out)
    ctx.deregister_table("rm_c2")


def c3(ctx, dev, scale, steps, out):
    n = int(25_000_000 * scale)
    g = torch.Generator(device=dev)
    g.manual_seed(42 + 3)
    offs, data, v, _, total = make_strings(n, g, dev)
    ctx.register_device_table("rm_pii", {"s": dict(dtype=F.TG_UTF8, n_rows=n, values=data.data_ptr(), offsets=offs.data_ptr(),
                                                   validity=v.data_ptr(), n_value_bytes=total)}, keepalive=[offs, data, v])
    lib = F.lib()

    def slots(p):
        return [lib.tg_plan_add_format(p.handle, b"s", 0, b"@", 0, 0.5, None), lib.tg_plan_add_format(p.handle, b"s", 1, None, 0, 0.5, None),
                lib.tg_plan_add_format(p.handle, b"s", 11, None, 0, 0.05, None), lib.tg_plan_add_format(p.handle, b"s", 3, None, 1, 0.5, None)]
    res = alternate({"off": build(slots, False), "on": build(slots, True)}, ctx, "rm_pii", steps)
    line("c3_string_formats", n, 4, res, out)
    ctx.deregister_table("rm_pii")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_row_masks: no CUDA device (nothing is measured without one)")
    dev = torch.device("cuda", 0)
    ctx = T.SessionContext(0)
    try:
        c2(ctx, dev, a.scale, a.steps, a.out)
        c3(ctx, dev, a.scale, a.steps, a.out)
    finally:
        ctx.close()


if __name__ == "__main__":
    main()
