#!/usr/bin/env python3
"""Cost of key-level row verdicts (tg_plan_request_key_rows) on the C4 shapes: is_unique over 125 M Int64 keys, dense
(a permutation: the bitmap path) and sparse (ids spread over 64 bits: the sorted-bucket path), each with the C4 1e-6
duplicates and with none (the fast exit: no row pass against the repeated-key table), and the 125 M -> 12.5 M foreign key.
Each plan runs without and with a request (DUPLICATE + FIRST, or ORPHAN), alternating step by step. Prints one JSON line per
workload: mean device ms of both arms (the plan's gpu_ms), the bytes the verdict arrays write, and the card's name and
power limit.

    python tools/bench_key_rows.py [--steps 10] [--scale 1.0] [--out key_rows.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import term_b200 as T  # noqa: E402
from term_b200 import _ffi as F  # noqa: E402
from tools.bench_row_masks import alternate, card  # noqa: E402
from tools.bench_suites import validity  # noqa: E402


def line(name, n, arrays, res, extra, out):
    off, on = res["off"], res["on"]
    rec = {"workload": name, "rows": n, "gpu_ms_off": off[0], "gpu_ms_on": on[0], "wall_ms_off": off[1], "wall_ms_on": on[1],
           "gpu_overhead": on[0] / off[0] - 1.0, "verdict_bytes_written": arrays * 2 * ((n + 31) // 32) * 4, "card": card()}
    rec.update(extra)
    print(json.dumps(rec), flush=True)
    if out:
        with open(out, "a") as f:
            f.write(json.dumps(rec) + "\n")


def uniq_plans(col):
    lib, A = F.lib(), F.tg_assertion(0, 0.0, 0.0)
    plans = {}
    for arm in ("off", "on"):
        p = T.api.Plan()
        s = lib.tg_plan_add_uniqueness(p.handle, (C.c_char_p * 1)(col.encode()), 1, 0, 0.9, A, 0)
        if arm == "on":
            p.request_key_rows(s, F.TG_KEY_ROWS_DUPLICATE)
            p.request_key_rows(s, F.TG_KEY_ROWS_FIRST)
        plans[arm] = p
    return plans, s


def is_unique(ctx, dev, n, steps, out, sparse, dups):
    g = torch.Generator(device=dev)
    g.manual_seed(42 + 4)
    keys = torch.randperm(n, generator=g, device=dev, dtype=torch.int64)
    if sparse:
        keys = (keys * 1_000_003) ^ 0x5DEECE66D
    if dups:
        ndup = max(1, n // 1_000_000)
        keys[torch.randint(0, n, (ndup,), generator=g, device=dev)] = keys[torch.randint(0, n, (ndup,), generator=g, device=dev)]
    v = validity(n, g, dev, 0.01)
    ctx.register_device_table("kr_keys", {"k": dict(dtype=F.TG_INT64, n_rows=n, values=keys.data_ptr(), validity=v.data_ptr())},
                              keepalive=[keys, v])
    plans, s = uniq_plans("k")
    res = alternate(plans, ctx, "kr_keys", steps)
    r = plans["on"].result(s)
    name = "c4_is_unique" + ("_sparse" if sparse else "") + ("" if dups else "_no_duplicates")
    line(name, n, 2, res, {"metric": r.metric, "metric_off": plans["off"].result(s).metric}, out)
    ctx.deregister_table("kr_keys")


def foreign_key(ctx, dev, n, steps, out):
    g = torch.Generator(device=dev)
    g.manual_seed(42 + 4)
    m = max(1000, n // 10)
    parent = torch.randperm(m, generator=g, device=dev, dtype=torch.int64)
    child = torch.randint(0, int(m * (1 + 1e-4)), (n,), generator=g, device=dev, dtype=torch.int64)
    cv = validity(n, g, dev, 0.01)
    ctx.register_device_table("kr_customers", {"id": dict(dtype=F.TG_INT64, n_rows=m, values=parent.data_ptr(), validity=None)},
                              keepalive=[parent])
    ctx.register_device_table("kr_orders", {"customer_id": dict(dtype=F.TG_INT64, n_rows=n, values=child.data_ptr(),
                                                                  validity=cv.data_ptr())}, keepalive=[child, cv])
    plans = {}
    for arm in ("off", "on"):
        p = T.api.Plan()
        s = F.lib().tg_plan_add_foreign_key(p.handle, b"kr_orders.customer_id", b"kr_customers.id", 0, 100)
        if arm == "on":
            p.request_key_rows(s, F.TG_KEY_ROWS_ORPHAN)
        plans[arm] = p
    res = alternate(plans, ctx, "kr_orders", steps)
    line("c4_foreign_key", n, 1, res, {"parent_rows": m, "metric": plans["on"].result(s).metric,
                                       "metric_off": plans["off"].result(s).metric}, out)
    ctx.deregister_table("kr_orders")
    ctx.deregister_table("kr_customers")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_key_rows: no CUDA device (nothing is measured without one)")
    dev = torch.device("cuda", 0)
    n = int(125_000_000 * a.scale)
    ctx = T.SessionContext(0)
    try:
        for sparse in (False, True):
            for dups in (True, False):
                is_unique(ctx, dev, n, a.steps, a.out, sparse, dups)
        foreign_key(ctx, dev, n, a.steps, a.out)
    finally:
        ctx.close()


if __name__ == "__main__":
    main()
