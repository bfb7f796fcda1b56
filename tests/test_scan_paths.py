"""The fused numeric scan (K1) through every plan shape, against an exact reference.

The planner picks, per scan pass, a tile (4096 rows, halved until the pass's shared-memory ring fits), a number of
units (each aggregate replicated over row slices of the tile until there are as many units as consumer warps) and
where unit state lives (registers, or per-lane shared memory when a pass has more units than warps). The knobs
TG_SCAN_TILE_ROWS, TG_SCAN_UNITS and TG_SCAN_MIN_STAGES are read on every execute; each case below sets them, restates
the planner's choice in Python (`planned_shape`) and asserts from the plan's exec stats that the scan ran that shape.

References are exact and computed here: Python ints for counts, Int64 MIN / MAX / wrapping SUM (compared bit for bit
in the aggregate's partial state); math.fsum for float sums and means; the two-pass fsum form for VARIANCE / STDDEV /
COVAR / CORR; numpy with SQL three-valued logic for predicate counts, cross-checked against the oracle's SQL evaluator.

Tolerances come from the error bound of the shifted sums (DESIGN.md, K1): with K an element of the column,
m2 = Σ(x-K)² - (Σ(x-K))²/n loses at most (L + 3)·eps·(Σ(x-K)² + (Σ(x-K))²/n) for chains of length L <= n, and for
data whose pivot lies within a few standard deviations of the mean both terms are at most ~10·m2. So a relative error
of MOMENT_C·(n + 16)·eps with MOMENT_C = 32 holds for every well-pivoted column and fails by many orders of magnitude
when K = 0 under a large mean (1e8 ± 1 loses every digit). Means and float sums are bounded by 1e-12·Σ|x| (a sum of n
values in chains of length L errs by at most L·eps·Σ|x|; 1e-12 is ~4500·eps, far above the L the planner produces).
"""
import math
import struct

import numpy as np
import pyarrow as pa
import pytest

from oracle import term_oracle as O

EPS = 2.0 ** -52
MOMENT_C = 32
SUM_REL = 1e-12
INT64_MIN, INT64_MAX = -(1 << 63), (1 << 63) - 1
MASK64 = (1 << 64) - 1
A_VALID, A_NUM, A_PAIR, A_PRED = 1, 2, 3, 4

# ------------------------------------------------------------------------------------------ the planner, restated ----
SCAN_TABLES_BYTES = 7168                       # sizeof(ScanTables) (scan_defs.h)
SMEM_BUDGET = 227 * 1024 - 256 - SCAN_TABLES_BYTES
CONSUMER_WARPS, STATE_SLOTS, MAX_STAGES = 16, 8, 8

SHAPES = {
    "default": {},
    "tile128": {"TG_SCAN_TILE_ROWS": "128"},
    "tile1024": {"TG_SCAN_TILE_ROWS": "1024"},
    "units1": {"TG_SCAN_UNITS": "1"},
    "units5": {"TG_SCAN_UNITS": "5"},
    "units40": {"TG_SCAN_UNITS": "40"},
    "stages2": {"TG_SCAN_MIN_STAGES": "2"},
}
SCAN_ENV = ("TG_SCAN_TILE_ROWS", "TG_SCAN_UNITS", "TG_SCAN_MIN_STAGES")


def _set_shape(monkeypatch, shape):
    for v in SCAN_ENV:
        monkeypatch.delenv(v, raising=False)
    for k, v in SHAPES[shape].items():
        monkeypatch.setenv(k, v)


def _ru(x, a):
    return (x + a - 1) // a * a


def planned_pass(shape, n_ops, n_count, cols):
    """(tile rows, units) of one pass as run_scan_pass picks them; cols: [(need_values, is_bool, has_bitmap)]"""
    env = SHAPES[shape]
    tile = max(128, int(env["TG_SCAN_TILE_ROWS"]) // 128 * 128) if "TG_SCAN_TILE_ROWS" in env else 4096
    target = min(48, max(1, int(env.get("TG_SCAN_UNITS", CONSUMER_WARPS))))
    min_stages = max(2, int(env.get("TG_SCAN_MIN_STAGES", 3)))
    while tile >= 128:
        chunks = tile // 128
        units = max(n_ops, min(target, n_count + (n_ops - n_count) * chunks))
        state = 0 if units <= CONSUMER_WARPS else units * STATE_SLOTS * 32 * 8
        stage = sum((_ru(tile // 8 if b else tile * 8, 128) if v else 0) + (_ru(tile // 8, 128) if bm else 0) for v, b, bm in cols) or 128
        if state + min_stages * stage + 2 * MAX_STAGES * 8 <= SMEM_BUDGET:
            return tile, units
        tile //= 2
    raise AssertionError("no tile fits")


def planned_shape(shape, ops, bitmap, dtypes):
    """expected exec stats of a plan: ops = [(first column, is_count, {column: needs values})] in the order the plan
    holds them; passes are formed as exec_scan_jobs forms them (stable sort by the first column's ordinal, at most
    16 aggregates per pass)"""
    order = list(dtypes)
    ops = sorted(ops, key=lambda o: order.index(o[0]))
    passes = [ops[k:k + CONSUMER_WARPS] for k in range(0, len(ops), CONSUMER_WARPS)]
    tiles, units = [], []
    for p in passes:
        cols = {}
        for _, _, used in p:
            for c, v in used.items():
                cols[c] = cols.get(c, False) or v
        t, u = planned_pass(shape, len(p), sum(1 for o in p if o[1]),
                            [(v, dtypes[c] == "bool", bitmap[c]) for c, v in cols.items()])
        tiles.append(t)
        units.append(u)
    return {"scan_passes": len(passes), "scan_min_tile_rows": min(tiles), "scan_max_units": max(units),
            "scan_smem_state": int(max(units) > CONSUMER_WARPS)}


def _assert_shape(plan, want):
    st = plan.stats()
    got = {k: st[k] for k in want}
    assert got == want, (got, want)


# ------------------------------------------------------------------------------------------------- plumbing ----
def _states(plan):
    """the partial state of every aggregate, keyed like plan.aggregates(): (kind, err, u[8] as uint64, f[8])"""
    blob = plan.partial_export()
    (n,) = struct.unpack_from("<Q", blob, 0)
    p, out = 8, {}
    keys = plan.aggregates()
    for i in range(n):
        kind, err = struct.unpack_from("<QQ", blob, p)
        u = struct.unpack_from("<8Q", blob, p + 16)
        f = struct.unpack_from("<8d", blob, p + 80)
        p += 144
        (bl,) = struct.unpack_from("<Q", blob, p)
        p += 8 + _ru(bl, 8)
        (ml,) = struct.unpack_from("<Q", blob, p)
        p += 8 + _ru(ml, 8)
        out[keys[i][1]] = (kind, err, u, f)
    return out


def _s64(u):
    return u - (1 << 64) if u >= (1 << 63) else u


def _run(ctx, table, constraints):
    import term_b200 as T
    plan = T.Plan()
    slots = [c._add_to(plan) for c in constraints]
    plan.execute(ctx, table)
    return plan, [c._result(plan, s) for c, s in zip(constraints, slots)]


def _bitmaps(ctx, table, names):
    return {c: bool(ctx.column_buffers(table, c)["validity"]) for c in names}


# ------------------------------------------------------------------------------------------------ reference ----
def ref_num(v, valid, integer):
    x = v[valid]
    n = len(x)
    r = {"n": n}
    if n == 0:
        return r
    xf = x.astype(np.float64)
    if integer:
        x64 = x.astype(np.int64)
        s = int((x64 >> 32).sum()) * (1 << 32) + int((x64 & 0xFFFFFFFF).sum())  # exact: both halves sum within int64
        r.update(min=int(x.min()), max=int(x.max()), isum=s & MASK64, mean=s / n, sum_abs=float(np.abs(xf).sum()))
    else:
        r.update(min=float(x.min()), max=float(x.max()), sum=math.fsum(xf.tolist()), sum_abs=math.fsum(np.abs(xf).tolist()))
        r["mean"] = r["sum"] / n
    if n >= 2:
        m = math.fsum(xf.tolist()) / n
        r["var"] = math.fsum(((xf - m) ** 2).tolist()) / (n - 1)
    return r


def ref_pair(x, vx, y, vy):
    m = vx & vy
    a, b = x[m].astype(np.float64), y[m].astype(np.float64)
    n = len(a)
    if n < 3:
        return {"n": n}
    da, db = a - math.fsum(a.tolist()) / n, b - math.fsum(b.tolist()) / n
    sxx, syy, sxy = math.fsum((da * da).tolist()), math.fsum((db * db).tolist()), math.fsum((da * db).tolist())
    return {"n": n, "cov": sxy / (n - 1), "corr": sxy / math.sqrt(sxx * syy) if sxx > 0 and syy > 0 else None,
            "sx": math.sqrt(sxx / (n - 1)), "sy": math.sqrt(syy / (n - 1))}


def moment_tol(n):
    return MOMENT_C * (n + 16) * EPS


def check_mean_sum(got, ref, what):
    assert got is not None, what
    assert abs(got - ref["mean"]) <= SUM_REL * ref["sum_abs"] / ref["n"], (what, got, ref["mean"])


def check_var(got, ref, what, stddev=False):
    want = math.sqrt(ref["var"]) if stddev else ref["var"]
    assert got is not None, what
    assert abs(got - want) <= moment_tol(ref["n"]) * want, (what, got, want, abs(got - want) / max(want, 1e-300))


# ------------------------------------------------------------------------------------------- the scan matrix ----
# columns (ordinal order) and what each one exercises
DTYPES = {"i": "i64", "f": "f64", "g": "f64", "k": "i64", "j": "i64", "w": "i32", "h": "f32", "b": "bool", "z": "i64"}
NUMERIC = {"i": "i", "f": "f", "g": "f", "k": "i", "j": "i", "w": "i", "h": "f", "z": "i"}


def matrix_columns(n, tile, seed):
    """name -> (values, valid): i Int64 over ±2^62 with INT64_MIN / INT64_MAX, sparse NULLs; f Float64 1e8 ± 1 with sparse
    NULLs and an all-NULL tile in the middle; g Float64 without bitmap; k Int64 1.7e12 ± 1000 after a leading NULL run
    (70,000 rows, or 3/4 of a smaller table); j Int64 without bitmap; w Int32, h Float32 (widened views, no bitmap);
    b Boolean, sparse NULLs; z all NULL. NULL slots hold values too (the scan must mask them)."""
    rng = np.random.default_rng(seed)

    def sparse():
        valid = rng.random(n) >= 0.05
        valid[n // 2] = False
        return valid

    i = rng.integers(-2 ** 62, 2 ** 62, n, dtype=np.int64)
    vi = sparse()
    if n >= 4:
        i[[1, n - 2]] = [INT64_MIN, INT64_MAX]
        vi[[1, n - 2]] = True
        i[n // 2] = INT64_MIN  # under a NULL
    f = 1e8 + rng.uniform(-1.0, 1.0, n)
    vf = sparse()
    if n > 2 * tile:
        vf[tile:2 * tile] = False
    k = (1_700_000_000_000 + rng.integers(-1000, 1001, n)).astype(np.int64)
    vk = np.ones(n, dtype=bool)
    vk[:min(70_000, 3 * n // 4 if n > 1 else 1)] = False
    b = rng.random(n) < 0.5
    return {
        "i": (i, vi), "f": (f, vf), "g": (rng.normal(0.0, 1.0, n), None), "k": (k, vk),
        "j": (rng.integers(-20, 21, n, dtype=np.int64), None), "w": (rng.integers(-1000, 1001, n).astype(np.int32), None),
        "h": (rng.normal(5.0, 2.0, n).astype(np.float32), None), "b": (b, sparse()), "z": (np.full(n, 7, dtype=np.int64), np.zeros(n, dtype=bool)),
    }


PA_TYPES = {"i64": pa.int64(), "f64": pa.float64(), "i32": pa.int32(), "f32": pa.float32(), "bool": pa.bool_()}


def _arrays(cols, lo, hi):
    return [pa.array(v[lo:hi], type=PA_TYPES[DTYPES[c]], mask=None if m is None else ~m[lo:hi]) for c, (v, m) in cols.items()]


def register(ctx, name, cols, n, how):
    """one batch; 8192-row batches; odd-length batches (validity boundaries off byte edges); a slice at offset 13"""
    names = list(cols)
    if how == "one":
        data = pa.table(_arrays(cols, 0, n), names=names)
    elif how == "b8192":
        data = [pa.RecordBatch.from_arrays(_arrays(cols, a, min(n, a + 8192)), names=names) for a in range(0, n, 8192)]
    elif how == "odd":
        data, a, lens = [], 0, [1, 7, 1001, 4099, 13, 70_001]
        while a < n:
            L = lens[len(data) % len(lens)]
            data.append(pa.RecordBatch.from_arrays(_arrays(cols, a, min(n, a + L)), names=names))
            a += L
    else:
        pad = {c: (np.concatenate([v[:1].repeat(13), v]), None if m is None else np.concatenate([np.ones(13, dtype=bool), m])) for c, (v, m) in cols.items()}
        data = pa.table(_arrays(pad, 0, n + 13), names=names).slice(13, n)
        assert data.column(0).chunks[0].offset == 13
    ctx.register_table(name, data)


# the big suite: more than 16 aggregates, so it runs as several passes; its first pass holds every aggregate whose first
# column is i, f or g and the rest go to the second (columns in brackets: the aggregate reads their values)
STATS = [("i", "Min"), ("i", "Max"), ("i", "Sum"), ("i", "Mean"), ("i", "StandardDeviation"),
         ("f", "Mean"), ("f", "Variance"), ("f", "Min"), ("f", "Max"), ("f", "Sum"),
         ("g", "Min"), ("g", "Max"),
         ("k", "Sum"), ("k", "StandardDeviation"), ("k", "Mean"),
         ("w", "Mean"), ("w", "StandardDeviation"), ("h", "Sum"), ("h", "Mean"), ("z", "Sum"), ("z", "Min"), ("j", "Sum")]
# (x, y, kind): every (Int64|Float64)² combination with 0, 1 and 2 bitmaps
PAIRS = [("g", "h", "corr"), ("j", "g", "cov"), ("h", "j", "corr"), ("j", "w", "cov"),
         ("f", "g", "corr"), ("i", "j", "cov"), ("i", "g", "corr"), ("f", "j", "cov"),
         ("f", "i", "cov"), ("i", "k", "corr"), ("k", "f", "cov")]
# (expression, first column, columns read {col: needs values}, numpy reference over the column dict)
PREDS = [
    ("i > 0", "i", {"i": True}, lambda c: _cmp(c, "i", ">", 0)),
    ("i >= 2.5", "i", {"i": True}, lambda c: _cmp(c, "i", ">=", 2.5)),
    ("f <= 100000000.5", "f", {"f": True}, lambda c: _cmp(c, "f", "<=", 100000000.5)),
    ("g <> 0.25 AND j < 10 AND i IS NOT NULL AND f = 100000000.0", "g", {"g": True, "j": True, "i": False, "f": True},
     lambda c: _cmp(c, "g", "<>", 0.25) & _cmp(c, "j", "<", 10) & c["i"][1] & _cmp(c, "f", "=", 1e8)),
    ("b IS NULL OR k < 1700000000000 OR g >= 1 OR j = 3", "b", {"b": False, "k": True, "g": True, "j": True},
     lambda c: ~c["b"][1] | _cmp(c, "k", "<", 1_700_000_000_000) | _cmp(c, "g", ">=", 1.0) | _cmp(c, "j", "=", 3)),
    ("j > 1", "j", {"j": True}, lambda c: _cmp(c, "j", ">", 1)),
    # forced into the predicate program
    ("j + 0 > 1", "j", {"j": True}, lambda c: _cmp(c, "j", ">", 1)),
    ("i % 7 = 0 OR f + g > 100000000.0", "i", {"i": True, "f": True, "g": True},
     lambda c: (c["i"][1] & (c["i"][0] % 7 == 0)) | (c["f"][1] & (c["f"][0] + c["g"][0] > 1e8))),
    ("CASE WHEN b THEN j ELSE 0 END > 10", "b", {"b": True, "j": True}, lambda c: c["b"][1] & c["b"][0] & (c["j"][0] > 10)),
    ("COALESCE(k, 0) > 1700000000000", "k", {"k": True}, lambda c: np.where(c["k"][1], c["k"][0], 0) > 1_700_000_000_000),
    ("b AND k > 1700000000000", "b", {"b": True, "k": True}, lambda c: c["b"][1] & c["b"][0] & _cmp(c, "k", ">", 1_700_000_000_000)),
]
# the small suite: few aggregates, so the planner replicates them over row slices (uneven for TG_SCAN_UNITS=5; more
# units than warps, state in shared memory, for TG_SCAN_UNITS=40)
SMALL_STATS = [("f", "Variance"), ("f", "Mean")]
SMALL_PAIRS = [("i", "k", "cov")]
SMALL_PREDS = [PREDS[0]]


def _cmp(c, name, op, lit):
    v, m = c[name]
    v = v.astype(np.float64) if isinstance(lit, float) else v
    r = {"<": v < lit, "<=": v <= lit, "=": v == lit, ">=": v >= lit, ">": v > lit, "<>": v != lit}[op]
    return r if m is None else (r & m)


def _suite(stats, pairs, preds, completeness):
    import term_b200 as T
    A = T.Assertion
    cons = [T.CompletenessConstraint(c, 0.5) for c in completeness]
    cons += [T.StatisticalConstraint(c, T.StatisticType[s], A.GreaterThan(-1e308)) for c, s in stats]
    cons += [(T.CorrelationConstraint.pearson if k == "corr" else T.CorrelationConstraint.covariance)(x, y, A.GreaterThan(-1e308)) for x, y, k in pairs]
    cons += [T.CustomSqlConstraint(e) for e, *_ in preds]
    return cons


def _suite_ops(stats, pairs, preds, completeness, bitmap):
    """the scan ops of a suite: COUNT(c) of a column without bitmap is answered on the host and one with a NUM
    aggregate on the same column is folded into it"""
    nums = []
    for c, _ in stats:
        if c not in nums:
            nums.append(c)
    ops = [(c, True, {c: False}) for c in completeness if bitmap[c] and c not in nums]
    ops += [(c, False, {c: True}) for c in nums]
    ops += [(x, False, {x: True, y: True}) for x, y, _ in pairs]
    ops += [(first, False, used) for _, first, used, _ in preds]
    return ops


def check_suite(ctx, table, cols, stats, pairs, preds, completeness, oracle_table=None):
    cons = _suite(stats, pairs, preds, completeness)
    plan, res = _run(ctx, table, cons)
    st = _states(plan)
    n = len(next(iter(cols.values()))[0])
    full = {c: (v, np.ones(n, dtype=bool) if m is None else m) for c, (v, m) in cols.items()}
    k = 0
    for c in completeness:
        nv = int(full[c][1].sum())
        assert res[k].metric == nv / n, (c, res[k].metric, nv, n)
        kind, err, u, _ = st["valid|" + c]
        assert err == 0 and u[1] == nv and u[0] == n, (c, u)
        k += 1
    nums = {}
    for c, s in stats:
        v, m = full[c]
        integer = NUMERIC[c] == "i"
        ref = nums.setdefault(c, ref_num(v, m, integer))
        g = res[k].metric
        kind, err, u, f = st["num|" + c]
        assert err == 0 and u[0] == ref["n"], (c, u[0], ref["n"])
        what = (c, s, n)
        if ref["n"] == 0 or (s in ("StandardDeviation", "Variance") and ref["n"] < 2):
            assert g is None, (what, g)
        elif s in ("Min", "Max"):
            want = ref["min" if s == "Min" else "max"]
            if integer:
                assert _s64(u[2 if s == "Min" else 3]) == want, what  # bit for bit in the state
            else:
                assert f[3 if s == "Min" else 4] == want, what
            assert g == float(want), (what, g, want)
        elif s == "Sum" and integer:
            if DTYPES[c] == "i64":
                assert u[1] == ref["isum"], what  # the wrapping sum mod 2^64, bit for bit
            assert g == float(_s64(ref["isum"])), (what, g)
        elif s == "Sum":
            assert abs(g - ref["sum"]) <= SUM_REL * ref["sum_abs"], (what, g, ref["sum"])
        elif s == "Mean":
            check_mean_sum(g, ref, what)
        else:
            check_var(g, ref, what, stddev=s == "StandardDeviation")
        k += 1
    for x, y, kind in pairs:
        ref = ref_pair(full[x][0], full[x][1], full[y][0], full[y][1])
        _, err, u, _ = st[f"pair|{x}|{y}"]
        assert err == 0 and u[0] == ref["n"], (x, y, u[0], ref["n"])
        g = res[k].metric
        if ref["n"] >= 3:
            if kind == "cov":
                assert abs(g - ref["cov"]) <= moment_tol(ref["n"]) * ref["sx"] * ref["sy"], (x, y, g, ref["cov"])
            elif ref["corr"] is not None:
                assert abs(g - ref["corr"]) <= 2 * moment_tol(ref["n"]), (x, y, g, ref["corr"])
        k += 1
    for expr, _, _, fn in preds:
        want = int(np.count_nonzero(fn(full)))
        _, err, u, _ = st["pred|" + expr]
        assert err == 0 and u[0] == want and u[1] == 0 and u[2] == n, (expr, u[:3], want)
        assert res[k].metric == want / n, (expr, res[k].metric, want)
        if oracle_table is not None:
            o = O.custom_sql(oracle_table, expr)
            assert (res[k].status.name.lower(), res[k].metric, res[k].message) == (o.status, o.metric, o.message), expr
        k += 1
    assert k == len(res)
    return plan


def _matrix_tile(shape):
    """the tile of the small suite's one pass (three aggregates over i, f, k, all with bitmaps): the row counts of a case
    are placed around it"""
    return planned_pass(shape, 3, 0, [(True, False, True)] * 3)[0]


def _rows(shape, which):
    t = _matrix_tile(shape)
    return {"1": 1, "31": 31, "127": 127, "128": 128, "129": 129, "tile-1": t - 1, "tile+1": t + 1,
            "148tile-1": 148 * t - 1, "148tile+1": 148 * t + 1, "several": 3 * 148 * t + t // 2 + 3}[which]


ALL_ROWS = ["1", "31", "127", "128", "129", "tile-1", "tile+1", "148tile-1", "148tile+1", "several"]
MATRIX = ([("default", r, how) for r in ALL_ROWS for how in ("one", "b8192", "odd", "slice")]
          + [(s, r, how) for s in SHAPES if s != "default" for r in ("129", "tile+1", "148tile+1") for how in ("one", "odd")]
          + [(s, "several", how) for s in ("tile128", "units40") for how in ("one", "odd")])


@pytest.mark.gpu
@pytest.mark.parametrize("shape,rows,how", MATRIX)
def test_scan_matrix(ctx, monkeypatch, shape, rows, how):
    """every aggregate kind of K1 over the plan shape `shape`, the row count `rows` (relative to the tile the planner
    picks) and the registration `how`, against the exact reference; the exec stats prove the shape ran"""
    _set_shape(monkeypatch, shape)
    n = _rows(shape, rows)
    cols = matrix_columns(n, _matrix_tile(shape), seed=n)
    name = f"scan_{shape}_{rows}_{how}".replace("+", "p").replace("-", "m")
    register(ctx, name, cols, n, how)
    try:
        bitmap = _bitmaps(ctx, name, DTYPES)
        assert not any(bitmap[c] for c in "gjwh") and all(bitmap[c] for c in "ifkbz"), bitmap
        oracle_table = pa.table(_arrays(cols, 0, n), names=list(cols)) if how == "one" and shape == "default" and n <= 20_000 else None
        plan = check_suite(ctx, name, cols, STATS, PAIRS, PREDS, ["b", "z", "i"], oracle_table)
        _assert_shape(plan, planned_shape(shape, _suite_ops(STATS, PAIRS, PREDS, ["b", "z", "i"], bitmap), bitmap, DTYPES))
        plan = check_suite(ctx, name, cols, SMALL_STATS, SMALL_PAIRS, SMALL_PREDS, [])
        want = planned_shape(shape, _suite_ops(SMALL_STATS, SMALL_PAIRS, SMALL_PREDS, [], bitmap), bitmap, DTYPES)
        assert want["scan_min_tile_rows"] == _matrix_tile(shape)
        _assert_shape(plan, want)
        if shape == "units5":
            assert want["scan_max_units"] == 5  # three aggregates over five row slices: uneven replication
        if shape == "units40":
            assert want["scan_smem_state"] == 1
    finally:
        ctx.deregister_table(name)


@pytest.mark.gpu
def test_scan_deterministic(ctx, monkeypatch):
    """the same suite executed twice on the same table gives bit-identical states (fixed-order reduction of the per-CTA
    partials), in registers and with shared-memory state"""
    n = 3 * 148 * 1024 + 77
    cols = matrix_columns(n, 1024, seed=5)
    register(ctx, "scan_det", cols, n, "b8192")
    try:
        for shape in ("default", "units40"):
            _set_shape(monkeypatch, shape)
            blobs = []
            for _ in range(2):
                import term_b200 as T
                plan = T.Plan()
                for c in _suite(STATS, PAIRS, PREDS, ["b", "z", "i"]):
                    c._add_to(plan)
                plan.execute_partial(ctx, "scan_det")
                blobs.append(plan.partial_export())
            assert blobs[0] == blobs[1], shape
    finally:
        ctx.deregister_table("scan_det")


# ---------------------------------------------------------------------------------------- values at the edges ----
def _stat_results(ctx, name, col, stats):
    import term_b200 as T
    cons = [T.StatisticalConstraint(col, T.StatisticType[s], T.Assertion.LessThan(1e300)) for s in stats]
    return _run(ctx, name, cons)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["default", "tile128"])
def test_nan_and_inf_propagate(ctx, monkeypatch, shape):
    """SUM / MEAN / STDDEV / VARIANCE of a column holding one NaN are NaN; with one +inf SUM and MEAN are +inf and
    STDDEV / VARIANCE NaN (inf - inf), as DataFusion computes them; the oracle agrees. The NaN sits in the first row,
    so the pivot has to skip it."""
    import term_b200 as T
    _set_shape(monkeypatch, shape)
    n = 10_000
    rng = np.random.default_rng(11)
    base = rng.normal(50.0, 3.0, n)
    x_nan, x_inf = base.copy(), base.copy()
    x_nan[0] = np.nan
    x_inf[n // 3] = np.inf
    t = pa.table({"xn": pa.array(x_nan), "xi": pa.array(x_inf, mask=np.arange(n) % 17 == 5)})
    ctx.register_table("scan_nan", t)
    try:
        stats = ["Sum", "Mean", "StandardDeviation", "Variance"]
        for col, want in (("xn", [math.nan] * 4), ("xi", [math.inf, math.inf, math.nan, math.nan])):
            plan, res = _stat_results(ctx, "scan_nan", col, stats)
            for s, r, w in zip(stats, res, want):
                o = O.statistic(t, col, s, ("LessThan", 1e300))
                assert r.metric is not None and (math.isnan(r.metric) if math.isnan(w) else r.metric == w), (col, s, r.metric)
                assert o.metric is not None and (math.isnan(o.metric) if math.isnan(w) else o.metric == w), (col, s, o.metric)
                assert r.status.name.lower() == o.status == "failure", (col, s, r.status, o.status)
        # has_standard_deviation(c, LessThan(x)) must not pass on a column holding NaN
        r = T.StatisticalConstraint("xn", T.StatisticType.StandardDeviation, T.Assertion.LessThan(100.0)).evaluate(ctx, "scan_nan")
        assert r.status.name == "Failure" and math.isnan(r.metric)
        a = T.StandardDeviationAnalyzer("xi").compute(ctx, "scan_nan")
        assert a.map["mean"] == math.inf and math.isnan(a.map["std_dev"]) and math.isnan(a.map["variance"])
        assert math.isnan(a.map["sample_variance"]) and math.isnan(a.map["coefficient_of_variation"])
    finally:
        ctx.deregister_table("scan_nan")


@pytest.mark.gpu
def test_variance_beyond_double_range_is_inf(ctx):
    """finite values whose variance exceeds the double range (normal(0, 1e3) with every 7th value 1e300): VARIANCE and
    STDDEV are +inf (DataFusion's accumulator overflows the same way), not NaN and not 0; the exact variance, computed on
    the values scaled by 1e-300, confirms it is beyond DBL_MAX"""
    import term_b200 as T
    n = 20_000
    rng = np.random.default_rng(13)
    x = rng.normal(0.0, 1e3, n)
    x[::7] = 1e300
    valid = rng.random(n) > 0.05
    ctx.register_table("scan_big", pa.table({"c": pa.array(x, mask=~valid)}))
    try:
        scaled = ref_num(x * 1e-300, valid, False)
        assert math.log10(scaled["var"]) + 600 > math.log10(np.finfo(np.float64).max)
        _, res = _stat_results(ctx, "scan_big", "c", ["Variance", "StandardDeviation", "Mean"])
        assert res[0].metric == math.inf and res[1].metric == math.inf, (res[0], res[1])
        check_mean_sum(res[2].metric, ref_num(x, valid, False), ("c", "mean"))
        a = T.StandardDeviationAnalyzer("c").compute(ctx, "scan_big")
        assert a.map["std_dev"] == math.inf and a.map["sample_variance"] == math.inf
    finally:
        ctx.deregister_table("scan_big")


@pytest.mark.gpu
def test_subnormals_and_signed_zeros(ctx):
    """subnormal values and ±0.0: exact sums (every partial sum is a multiple of the smallest subnormal), exact MIN / MAX
    (the extremes are non-zero), moments within the bound"""
    n = 20_011
    rng = np.random.default_rng(3)
    x = rng.integers(-1000, 1001, n).astype(np.float64) * 5e-324
    x[::7] = 0.0
    x[3::7] = -0.0
    valid = rng.random(n) > 0.1
    t = pa.table({"s": pa.array(x, mask=~valid)})
    ctx.register_table("scan_sub", t)
    try:
        ref = ref_num(x, valid, False)
        plan, res = _stat_results(ctx, "scan_sub", "s", ["Sum", "Mean", "Min", "Max", "Variance"])
        assert res[0].metric == ref["sum"] and res[2].metric == ref["min"] and res[3].metric == ref["max"]
        assert abs(res[1].metric - ref["mean"]) <= 5e-324
        assert abs(res[4].metric - ref["var"]) <= 5e-324  # the squares underflow to zero in both
    finally:
        ctx.deregister_table("scan_sub")


def _leading_null_table(n, lead, seed):
    rng = np.random.default_rng(seed)
    valid = np.ones(n, dtype=bool)
    valid[:lead] = False
    x = 1e8 + rng.uniform(-1.0, 1.0, n)
    y = 2.0 * x + rng.normal(0.0, 0.5, n)
    k = (1_700_000_000_000 + rng.integers(-1000, 1001, n)).astype(np.int64)
    w = (2_000_000_000 + rng.integers(-1000, 1001, n)).astype(np.int32)
    h = (10_000_000 + rng.integers(-1, 2, n)).astype(np.float32)
    cols = {"x": (x, valid), "y": (y, valid), "k": (k, valid), "w": (w, valid), "h": (h, valid)}
    types = {"x": pa.float64(), "y": pa.float64(), "k": pa.int64(), "w": pa.int32(), "h": pa.float32()}
    t = pa.table({c: pa.array(v, type=types[c], mask=~m) for c, (v, m) in cols.items()})
    return t, cols


def _check_large_mean(ctx, name, cols):
    import term_b200 as T
    A = T.Assertion
    cons = [T.StatisticalConstraint(c, T.StatisticType[s], A.GreaterThan(-1e308)) for c in cols for s in ("Variance", "StandardDeviation", "Mean")]
    cons += [T.CorrelationConstraint.pearson("x", "y", A.GreaterThan(-2.0)), T.CorrelationConstraint.covariance("x", "y", A.GreaterThan(-1e308)),
             T.CorrelationConstraint.covariance("k", "w", A.GreaterThan(-1e308))]
    plan, res = _run(ctx, name, cons)
    k = 0
    for c, (v, m) in cols.items():
        ref = ref_num(v, m, v.dtype.kind == "i")
        check_var(res[k].metric, ref, (c, "var"))
        check_var(res[k + 1].metric, ref, (c, "stddev"), stddev=True)
        check_mean_sum(res[k + 2].metric, ref, (c, "mean"))
        k += 3
    for x, y, kind in (("x", "y", "corr"), ("x", "y", "cov"), ("k", "w", "cov")):
        ref = ref_pair(cols[x][0], cols[x][1], cols[y][0], cols[y][1])
        g = res[k].metric
        if kind == "corr":
            assert abs(g - ref["corr"]) <= 2 * moment_tol(ref["n"]), (x, y, g, ref["corr"])
        else:
            assert abs(g - ref["cov"]) <= moment_tol(ref["n"]) * ref["sx"] * ref["sy"], (x, y, g, ref["cov"])
        k += 1
    a = T.StandardDeviationAnalyzer("x").compute(ctx, name)
    ref = ref_num(cols["x"][0], cols["x"][1], False)
    assert abs(a.map["sample_variance"] - ref["var"]) <= moment_tol(ref["n"]) * ref["var"], (a.map, ref["var"])


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["one", "b8192"])
def test_leading_null_run_keeps_pivot_an_element(ctx, how):
    """a column whose first 70,000 rows are NULL: appended as one batch, no head window holds a value, so the scan finds
    the pivot (in 8192-row batches the first batch with values sets it); large means with small spreads (Float64 1e8 ± 1, Int64 1.7e12 ± 1000, Int32 2e9 ± 1000, Float32 1e7 ± 1)
    must meet the same moment bound as well-centred data"""
    n = 200_000
    t, cols = _leading_null_table(n, 70_000, seed=21)
    name = f"scan_lead_{how}"
    ctx.register_table(name, t if how == "one" else t.to_batches(max_chunksize=8192))
    try:
        _check_large_mean(ctx, name, cols)
    finally:
        ctx.deregister_table(name)


@pytest.mark.gpu
def test_parquet_leading_null_run(ctx, tmp_path):
    """a Parquet row group that starts with 5,000 NULLs (the decoder takes the pivot from a chunk's first 4096 values)"""
    import pyarrow.parquet as pq
    n = 60_000
    t, cols = _leading_null_table(n, 5_000, seed=22)
    path = tmp_path / "lead.parquet"
    pq.write_table(t, path, row_group_size=n, compression="NONE", use_dictionary=False)
    ctx.register_parquet("scan_lead_pq", str(path))
    try:
        _check_large_mean(ctx, "scan_lead_pq", cols)
    finally:
        ctx.deregister_table("scan_lead_pq")


# ------------------------------------------------------------------------------------ predicates at the edges ----
OPS = ["<", "=", "<=", ">", ">=", "<>"]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["default", "tile128", "units40"])
def test_terms_every_operator(ctx, monkeypatch, shape):
    """TERMS units: each comparison on Int64 against an integer literal, on Float64 against a float literal and on Int64
    against a float literal (compared as Float64), IS [NOT] NULL, AND / OR of up to four terms; numpy with SQL
    three-valued logic as the reference and the oracle's evaluator as a cross-check"""
    import term_b200 as T
    _set_shape(monkeypatch, shape)
    n = 20_003
    rng = np.random.default_rng(4)
    a = rng.integers(-40, 41, n, dtype=np.int64)
    a[:3] = [INT64_MIN, INT64_MAX, 17]
    x = rng.uniform(-2.0, 2.0, n).round(1)
    va, vx = rng.random(n) > 0.1, rng.random(n) > 0.2
    va[:3] = True
    t = pa.table({"a": pa.array(a, mask=~va), "x": pa.array(x, mask=~vx)})
    c = {"a": (a, va), "x": (x, vx)}
    exprs = []
    for op in OPS:
        exprs += [(f"a {op} 17", _cmp(c, "a", op, 17)), (f"x {op} 0.5", _cmp(c, "x", op, 0.5)), (f"a {op} 16.5", _cmp(c, "a", op, 16.5)),
                  (f"17 {op} a", _cmp(c, "a", {"<": ">", ">": "<", "<=": ">=", ">=": "<="}.get(op, op), 17))]
    exprs += [("a IS NULL", ~va), ("x IS NOT NULL", vx),
              ("a > 0 AND x < 1.0", _cmp(c, "a", ">", 0) & _cmp(c, "x", "<", 1.0)),
              ("a > 0 OR x < 1.0", _cmp(c, "a", ">", 0) | _cmp(c, "x", "<", 1.0)),
              ("a > 0 AND x < 1.0 AND a <> 5 AND x IS NOT NULL", _cmp(c, "a", ">", 0) & _cmp(c, "x", "<", 1.0) & _cmp(c, "a", "<>", 5) & vx),
              ("a = 3 OR x = 0.5 OR a IS NULL OR x >= 1.5", _cmp(c, "a", "=", 3) | _cmp(c, "x", "=", 0.5) | ~va | _cmp(c, "x", ">=", 1.5))]
    ctx.register_table("scan_terms", t)
    try:
        cons = [T.CustomSqlConstraint(e) for e, _ in exprs]
        plan, res = _run(ctx, "scan_terms", cons)
        st = _states(plan)
        for (e, want), r in zip(exprs, res):
            _, err, u, _ = st["pred|" + e]
            assert err == 0 and u[0] == int(np.count_nonzero(want)), (e, u[0], int(np.count_nonzero(want)))
            o = O.custom_sql(t, e)
            assert (r.status.name.lower(), r.metric, r.message) == (o.status, o.metric, o.message), e
    finally:
        ctx.deregister_table("scan_terms")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["default", "tile128"])
def test_pred_programs(ctx, monkeypatch, shape):
    """the predicate register machine: arithmetic, `/` and `%` by zero (an error for the whole constraint), INT64_MIN / -1,
    CASE / COALESCE, a Boolean column and three-valued logic over NULLs, against the oracle; the same NaN-free predicate as
    TERMS (`c > 1`) and forced into the program (`c + 0 > 1`) counts the same rows"""
    import term_b200 as T
    _set_shape(monkeypatch, shape)
    n = 5_001
    rng = np.random.default_rng(9)
    a = rng.integers(-50, 51, n, dtype=np.int64)
    a[[0, 7]] = INT64_MIN
    z = rng.integers(0, 3, n, dtype=np.int64)
    x = rng.normal(0.0, 2.0, n)
    b = rng.random(n) < 0.5
    va, vz, vx, vb = (rng.random(n) > p for p in (0.1, 0.1, 0.15, 0.2))
    t = pa.table({"a": pa.array(a, mask=~va), "z": pa.array(z, mask=~vz), "x": pa.array(x, mask=~vx), "b": pa.array(b, mask=~vb)})
    exprs = ["a * 2 + 3 > x", "(a - 7) * (a + 7) < 100", "a / 0 > 1", "a % z = 1", "a / z > 2", "a / -1 > 0",
             "CASE WHEN b THEN a ELSE -a END > 10", "COALESCE(x, a, 0) > 0.5", "COALESCE(a, 1) % 2 = 0",
             "b", "NOT b", "b AND x > 0", "b OR x > 0", "NOT (a > 5)", "NOT (a > 5 AND x > 0)", "(a > 5) = (x > 0)",
             "a > 5 OR x IS NULL", "x > 1", "x + 0 > 1", "a > 1", "a + 0 > 1"]
    ctx.register_table("scan_pred", t)
    try:
        cons = [T.CustomSqlConstraint(e) for e in exprs]
        plan, res = _run(ctx, "scan_pred", cons)
        got = {}
        for e, r in zip(exprs, res):
            o = O.custom_sql(t, e)
            assert (r.status.name.lower(), r.metric, r.message) == (o.status, o.metric, o.message), (e, r, o)
            got[e] = r.metric
        assert got["x > 1"] == got["x + 0 > 1"] == np.count_nonzero(vx & (x > 1)) / n
        assert got["a > 1"] == got["a + 0 > 1"] == np.count_nonzero(va & (a > 1)) / n
        assert got["b AND x > 0"] == np.count_nonzero(vb & b & vx & (x > 0)) / n
        assert got["NOT (a > 5 AND x > 0)"] == np.count_nonzero((va & (a <= 5)) | (vx & (x <= 0))) / n
        assert res[exprs.index("a / 0 > 1")].metric is None
    finally:
        ctx.deregister_table("scan_pred")


# ------------------------------------------------------------------------------------------------ shard merge ----
@pytest.mark.gpu
def test_shard_merge_repivots(ctx):
    """two shards whose pivots differ by 1e8 merge through partial_merge (re-pivot onto the first shard's K) to the
    one-table answer within the same bound"""
    import term_b200 as T
    rng = np.random.default_rng(31)
    n = 100_000
    xa, xb = rng.normal(0.0, 1.0, n), 1e8 + rng.normal(0.0, 1.0, n)
    ya, yb = 0.5 * xa + rng.normal(0.0, 1.0, n), 0.5 * xb + rng.normal(0.0, 1.0, n)
    ka, kb = rng.integers(-1000, 1001, n, dtype=np.int64), (10 ** 8 + rng.integers(-1000, 1001, n)).astype(np.int64)
    va, vb = rng.random(n) > 0.05, rng.random(n) > 0.05
    mk = lambda x, y, k, v: pa.table({"x": pa.array(x, mask=~v), "y": pa.array(y), "k": pa.array(k, mask=~v)})
    ctx.register_table("shard_a", mk(xa, ya, ka, va))
    ctx.register_table("shard_b", mk(xb, yb, kb, vb))
    ctx.register_table("shard_ab", pa.concat_tables([mk(xa, ya, ka, va), mk(xb, yb, kb, vb)]))
    try:
        A = T.Assertion
        cons = [T.StatisticalConstraint(c, T.StatisticType[s], A.GreaterThan(-1e308)) for c in ("x", "k") for s in ("Variance", "Mean", "Sum", "Min")]
        cons += [T.CorrelationConstraint.pearson("x", "y", A.GreaterThan(-2.0)), T.CorrelationConstraint.covariance("k", "y", A.GreaterThan(-1e308))]
        plan = T.Plan()
        slots = [c._add_to(plan) for c in cons]
        parts = []
        for s in ("shard_a", "shard_b"):
            plan.execute_partial(ctx, s)
            parts.append(plan.partial_export())
        st = [_states_of(plan, p) for p in parts]
        assert abs(st[1]["num|x"][3][0] - st[0]["num|x"][3][0]) > 9e7  # the pivots differ by ~1e8
        plan.partial_reset()
        for p in parts:
            plan.partial_merge(p)
        plan.finalize()
        merged = [c._result(plan, s) for c, s in zip(cons, slots)]
        _, one = _run(ctx, "shard_ab", cons)
        v = np.concatenate([va, vb])
        x, y, k = np.concatenate([xa, xb]), np.concatenate([ya, yb]), np.concatenate([ka, kb])
        for res in (merged, one):
            i = 0
            for col, vals, integer in (("x", x, False), ("k", k, True)):
                ref = ref_num(vals, v, integer)
                check_var(res[i].metric, ref, (col, "var"))
                check_mean_sum(res[i + 1].metric, ref, (col, "mean"))
                want_sum = float(_s64(ref["isum"])) if integer else ref["sum"]
                assert abs(res[i + 2].metric - want_sum) <= SUM_REL * ref["sum_abs"], (col, res[i + 2].metric, want_sum)
                assert res[i + 3].metric == ref["min"]
                i += 4
            r = ref_pair(x, v, y, np.ones(2 * n, dtype=bool))
            assert abs(res[i].metric - r["corr"]) <= 2 * moment_tol(r["n"])
            r = ref_pair(k, v, y, np.ones(2 * n, dtype=bool))
            assert abs(res[i + 1].metric - r["cov"]) <= moment_tol(r["n"]) * r["sx"] * r["sy"]
    finally:
        for s in ("shard_a", "shard_b", "shard_ab"):
            ctx.deregister_table(s)


class _Blob:
    def __init__(self, plan, blob):
        self._p, self._b = plan, blob

    def aggregates(self):
        return self._p.aggregates()

    def partial_export(self):
        return self._b


def _states_of(plan, blob):
    return _states(_Blob(plan, blob))


# --------------------------------------------------------------------------------- finalize without a GPU ----
def _num_record(n, K, sd, sdd, sx):
    """one A_NUM shard state in the partial-blob layout: kind, err, u[8] (u0 = n), f[8] (f0 = K, f1 = Σd, f2 = Σd², f5 = Σx),
    empty blob, empty error message"""
    return (struct.pack("<QQ", A_NUM, 0) + struct.pack("<8Q", n, 0, 0, 0, 0, 0, 0, 0)
            + struct.pack("<8d", K, sd, sdd, 0.0, 0.0, sx, 0.0, 0.0) + struct.pack("<QQ", 0, 0))


@pytest.mark.parametrize("case", ["nan", "inf", "negative_m2", "overflow"])
def test_num_finalize_nan_and_rounding(built_lib, case):
    """STDDEV / VARIANCE finalize from merged shard states: NaN sums (a NaN or an infinite value in the column) give NaN,
    not 0, and a constraint on them fails; m2 pushed slightly below zero by rounding finalizes to 0, never negative;
    finite values whose squared deviations overflow (Σd finite, Σd² = +inf) give +inf, not inf - inf = NaN"""
    import term_b200.api as T
    cons = [T.StatisticalConstraint("c", T.StatisticType.StandardDeviation, T.Assertion.LessThan(10.0)),
            T.StatisticalConstraint("c", T.StatisticType.Variance, T.Assertion.LessThan(10.0))]
    an = T.StandardDeviationAnalyzer("c")
    plan = T.Plan()
    slots = [c._add_to(plan) for c in cons]
    aslot = an._add_to(plan)
    assert [k for k, _ in plan.aggregates()] == [A_NUM]
    if case == "nan":
        shards = [_num_record(3, 1.0, 0.5, 1.25, 3.5), _num_record(2, 2.0, math.nan, math.nan, math.nan)]
    elif case == "inf":
        shards = [_num_record(3, 1.0, 0.5, 1.25, 3.5), _num_record(2, 2.0, math.inf, math.inf, math.inf)]
    elif case == "negative_m2":
        # Σd = 3, Σd² = 3 - 2^-51 on n = 3: m2 = Σd² - (Σd)²/n = -2^-51 after rounding
        shards = [_num_record(3, 1.0, 3.0, 3.0 - 2.0 ** -51, 6.0)]
    else:
        # two values 1e300 and one 0 (K = 0): Σd = 2e300 is finite, Σd² and (Σd)²/n both overflow
        shards = [_num_record(3, 0.0, 2e300, math.inf, 2e300)]
    plan.partial_reset()
    for s in shards:
        plan.partial_merge(struct.pack("<Q", 1) + s)
    plan.finalize()
    r_sd, r_var = (c._result(plan, s) for c, s in zip(cons, slots))
    a = plan.analyzer_result(aslot)
    if case == "negative_m2":
        assert r_sd.metric == 0.0 and r_var.metric == 0.0 and r_sd.status.name == "Success"
        assert a.map["std_dev"] == 0.0 and a.map["variance"] == 0.0 and a.map["sample_variance"] == 0.0
    elif case == "overflow":
        assert r_sd.metric == math.inf and r_var.metric == math.inf and r_sd.status.name == "Failure"
        assert a.map["std_dev"] == math.inf and a.map["variance"] == math.inf and a.map["sample_variance"] == math.inf
    else:
        assert math.isnan(r_sd.metric) and math.isnan(r_var.metric), (r_sd, r_var)
        assert r_sd.status.name == "Failure" and r_var.status.name == "Failure"
        assert math.isnan(a.map["std_dev"]) and math.isnan(a.map["variance"]) and math.isnan(a.map["sample_std_dev"])


def test_oracle_variance_of_non_finite_columns():
    """the oracle's STDDEV / VARIANCE of a column holding NaN, +inf, or +inf and -inf together is NaN (math.fsum raises
    on the last), as DataFusion's"""
    for vals in ([1.0, math.nan, 2.0], [1.0, math.inf, 2.0], [math.inf, 1.0, -math.inf]):
        t = pa.table({"c": pa.array(vals)})
        for s in ("StandardDeviation", "Variance"):
            assert math.isnan(O.stat_value(O.table_cols(t)["c"], s)), (vals, s)
    t = pa.table({"c": pa.array([1.0, 2.0, 4.0])})
    assert O.stat_value(O.table_cols(t)["c"], "Variance") == 7.0 / 3.0
