"""Grouped completeness (K5) and the value histogram through every counting path, against an exact reference.

K5 has four ways to count a batch of groupings: the tile kernel (the default), the dictionary kernel (TG_GROUPED_NO_TILE),
marginal derivation of single-column groupings out of a composite one (on unless TG_GROUPED_NO_MARGINALS) and the 128-bit
fingerprint fallback (TG_GROUPED_NO_DICT, or whenever a CTA's dictionary / composite table overflows). Every case below runs
under each setting and must give the reference's groups and counts, identical across settings.

Two views are compared: the exact state (`execute_partial` + `partial_export`: key bytes, rows, non-NULL rows per group;
the only view that keeps NUL bytes in keys) and the finalized map (keys cross the C ABI as C strings). Key rendering is the
one of `run_grouped_batch`: Utf8 as raw bytes, integers in decimal, floats as Rust's `{}` after canonicalisation (-0.0 is
0.0, every NaN one group; which row represents a group is not pinned, so its zero may print as "-0"), Boolean as "" (as
"true" / "false" in a value histogram), NULL as "NULL" ("\\xffNULL" in a value histogram), fields joined by \\x1f."""
import struct
import time

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc
import pytest

from oracle import term_oracle as O

PATHS = {
    "default": {},
    "no_marginals": {"TG_GROUPED_NO_MARGINALS": "1"},
    "dict": {"TG_GROUPED_NO_TILE": "1"},
    "dict_no_marginals": {"TG_GROUPED_NO_TILE": "1", "TG_GROUPED_NO_MARGINALS": "1"},
    "fingerprint": {"TG_GROUPED_NO_DICT": "1"},
}
ENV_VARS = ("TG_GROUPED_NO_TILE", "TG_GROUPED_NO_DICT", "TG_GROUPED_NO_MARGINALS")
MAX_GROUPS = 1 << 20                    # GRP_MAX_GROUPS_DEV
LIMIT_MSG = "grouped completeness: more than 1048576 groups"
TG_ERR_UNSUPPORTED = 5
CTA_ROWS = 768                          # rows of one tile of the tile kernel
NULL_TAG1 = 0x9AE16A3B2F90404F          # the first word of a NULL's fingerprint pair (hash_common.cuh)
NULL_TAG1_I64 = int(np.array([NULL_TAG1], dtype=np.uint64).view(np.int64)[0])
NULL_TAG1_F64 = float(np.array([NULL_TAG1], dtype=np.uint64).view(np.float64)[0])
FLOAT_TYPES = (pa.float64(), pa.float32())


def _set_path(monkeypatch, path):
    for v in ENV_VARS:
        monkeypatch.delenv(v, raising=False)
    for k, v in PATHS[path].items():
        monkeypatch.setenv(k, v)


# ------------------------------------------------------------------------------------------------ reference ----
def _null_text(hist):
    return b"\xffNULL" if hist else b"NULL"


def _col_codes(arr, hist=False):
    """(codes, texts): per row the id of the value's group (-1: NULL), and per id the rendered key field"""
    if isinstance(arr, pa.ChunkedArray):
        arr = arr.combine_chunks()
    valid = np.asarray(arr.is_valid().to_numpy(zero_copy_only=False), dtype=bool)
    t = arr.type
    codes = np.full(len(arr), -1, dtype=np.int64)
    if pa.types.is_string(t):
        enc = pc.dictionary_encode(arr)
        codes = np.asarray(enc.indices.fill_null(-1).to_numpy(zero_copy_only=False), dtype=np.int64)
        return codes, enc.dictionary.cast(pa.binary()).to_pylist()
    if pa.types.is_boolean(t):
        vals = np.asarray(arr.fill_null(False).to_numpy(zero_copy_only=False), dtype=np.int64)
        codes[valid] = vals[valid]
        return codes, [b"false", b"true"] if hist else [b"", b""]
    if t in FLOAT_TYPES:
        bits = np.asarray(arr.fill_null(0.0).to_numpy(zero_copy_only=False), dtype=np.float64).view(np.uint64).copy()
        bits[(bits << np.uint64(1)) == 0] = 0                                   # -0.0 -> 0.0
        bits[np.isnan(bits.view(np.float64))] = np.uint64(0x7FF8000000000000)    # one NaN
        uniq, inv = np.unique(bits[valid], return_inverse=True)
        codes[valid] = inv
        return codes, [O.rust_f64(float(x)).encode() for x in uniq.view(np.float64)]
    vals = np.asarray(arr.fill_null(0).to_numpy(zero_copy_only=False)).astype(np.int64)
    uniq, inv = np.unique(vals[valid], return_inverse=True)
    codes[valid] = inv
    return codes, [str(int(x)).encode() for x in uniq]


def reference_groups(table, target, groups, hist=False, cache=None):
    """sorted [(key fields, rows, non-NULL target rows)]: one entry per group of values (Boolean groups render alike)"""
    cols = []
    for g in groups:
        if cache is not None and (g, hist) in cache:
            cols.append(cache[(g, hist)])
        else:
            cols.append(_col_codes(table.column(g), hist))
            if cache is not None:
                cache[(g, hist)] = cols[-1]
    tv = table.column(target)
    tv = np.asarray((tv.combine_chunks() if isinstance(tv, pa.ChunkedArray) else tv).is_valid().to_numpy(zero_copy_only=False), dtype=bool)
    bases = [len(texts) + 1 for _, texts in cols]
    assert float(np.prod(np.array(bases, dtype=np.float64))) < 2.0 ** 62
    key = np.zeros(len(tv), dtype=np.int64)
    for (codes, _), b in zip(cols, bases):
        key = key * b + (codes + 1)
    uniq, inv = np.unique(key, return_inverse=True)
    tot = np.bincount(inv, minlength=len(uniq))
    nn = np.bincount(inv[tv], minlength=len(uniq))
    digits = []
    rest = uniq.copy()
    for b in reversed(bases):
        digits.append(rest % b - 1)
        rest //= b
    digits.reverse()
    null = _null_text(hist)
    out = []
    for i in range(len(uniq)):
        out.append((tuple(texts[d[i]] if d[i] >= 0 else null for (_, texts), d in zip(cols, digits)), int(tot[i]), int(nn[i])))
    out.sort()
    return out


def reference_map(ref):
    """the finalized map: entries of equal rendered keys add up, fields joined by '_', ratio non-NULL / rows"""
    acc = {}
    for fields, t, n in ref:
        k = b"_".join(fields)
        a = acc.setdefault(k, [0, 0])
        a[0] += t
        a[1] += n
    return {k: n / t for k, (t, n) in acc.items()}


# ------------------------------------------------------------------------------------------------ exact state ----
def parse_partial(buf):
    """tg_plan_partial_export: [u64 n_aggs] then per aggregate kind, err, u[8], f[8], blob_len, blob, err_len, err (8-padded)"""
    (n,) = struct.unpack_from("<Q", buf, 0)
    off, out = 8, []
    for _ in range(n):
        kind, err = struct.unpack_from("<QQ", buf, off)
        off += 16 + 128
        (bl,) = struct.unpack_from("<Q", buf, off)
        blob = bytes(buf[off + 8: off + 8 + bl])
        off += 8 + ((bl + 7) & ~7)
        (ml,) = struct.unpack_from("<Q", buf, off)
        msg = bytes(buf[off + 8: off + 8 + ml]).decode()
        off += 8 + ((ml + 7) & ~7)
        out.append((kind, err, blob, msg))
    return out


def parse_groups(blob):
    """grouped state: [u64 n] then per group {u32 key_len, key, u64 rows, u64 non-NULL rows}"""
    (n,) = struct.unpack_from("<Q", blob, 0)
    off, out = 8, []
    mv = memoryview(blob)
    for _ in range(n):
        (L,) = struct.unpack_from("<I", blob, off)
        key = bytes(mv[off + 4: off + 4 + L])
        t, nn = struct.unpack_from("<QQ", blob, off + 4 + L)
        out.append((key, t, nn))
        off += 4 + L + 16
    assert off == len(blob)
    return out


def _float_fields(table, groups):
    return [table.schema.field(g).type in FLOAT_TYPES for g in groups]


def _norm_fields(fields, isf):
    return tuple(b"0" if f and x == b"-0" else x for x, f in zip(fields, isf))


def exact_groups(plan, key, table, groups):
    """(err, message, sorted [(key fields, rows, non-NULL rows)]) of aggregate `key` from the plan's exported state"""
    keys = [k for _, k in plan.aggregates()]
    _, err, blob, msg = parse_partial(plan.partial_export())[keys.index(key)]
    if err:
        return err, msg, None
    isf = _float_fields(table, groups)
    got = []
    for k, t, nn in parse_groups(blob):
        fields = tuple(k.split(b"\x1f")) if len(groups) > 1 else (k,)
        assert len(fields) == len(groups), k
        got.append((_norm_fields(fields, isf), t, nn))
    got.sort()
    return 0, "", got


def _map_compare(got_map, ref, table, groups):
    """the finalized map against the reference, leaving out keys a NUL byte makes ambiguous as C strings"""
    want = reference_map(ref)
    amb = {k.split(b"\0")[0] for k in want if b"\0" in k}
    isf = _float_fields(table, groups)
    got = {}
    for k, v in got_map.items():
        if k.startswith("__"):
            continue
        kb = k.encode()
        fields = tuple(kb.split(b"_")) if len(groups) > 1 else (kb,)
        kb = b"_".join(_norm_fields(fields, isf)) if len(fields) == len(groups) else kb
        got[kb] = v
    want = {k: v for k, v in want.items() if b"\0" not in k and k not in amb}
    got = {k: v for k, v in got.items() if k not in amb}
    assert got == want


# ------------------------------------------------------------------------------------------------ tables ----
LONG_A = ("long-" + "0123456789abcdefghijklmnopqrstuvwxyz" * 900)[:30000]
LONG_B = LONG_A[:-1] + "!"
S_POOL = ["", "a", "abcdefg", "abcdefgh", "abcdefghi", "abcdefghijklmno", "abcdefghijklmnop", "abcdefghijklmnopq", "x" * 100,
          "δέλτα", "日本語テキスト", "ab", "ab\0", "ab\0\0", "prefix08" + "-first", "prefix08" + "-other", "0123456789abcdef" + "-one",
          "0123456789abcdef" + "-two", "0123456789abcdef", "naïve café"]
I_POOL = [-(1 << 63), (1 << 63) - 1, -1, 0, NULL_TAG1_I64, 7, 123456789012]
NAN_A, NAN_B = np.array([0x7FF8000000000001, 0xFFF0000000000123], np.uint64).view(np.float64)  # two NaN payloads
F_POOL = [0.0, -0.0, NAN_A, NAN_B, np.inf, -np.inf, 5e-324, NULL_TAG1_F64, 1.5, -2.25]
I32_POOL = [-(1 << 31), (1 << 31) - 1, -5, 0, 42]
I8_POOL = [-128, 127, 0, -1]
U16_POOL = [0, 65535, 300]
F32_POOL = [0.5, -1.25, 3.0, 0.0, -0.0, 1024.125, 0.0078125]


def _pool_col(rng, pool, n, typ, null_rate):
    codes = rng.integers(0, len(pool), n)
    codes[: min(n, len(pool))] = np.arange(min(n, len(pool)))  # every pool value occurs
    mask = rng.random(n) < null_rate
    mask[: min(n, len(pool))] = False
    if pa.types.is_floating(typ):
        vals = np.array(pool, dtype=np.float64 if typ == pa.float64() else np.float32)[codes]
        return pa.array(vals, type=typ, mask=mask)
    if pa.types.is_integer(typ):
        return pa.array(np.array(pool, dtype=typ.to_pandas_dtype())[codes], type=typ, mask=mask)
    return pa.array(pool, type=typ).take(pa.array(codes, mask=mask))


def make_table(n, seed=11):
    rng = np.random.default_rng(seed)
    s = _pool_col(rng, S_POOL, n, pa.string(), 0.08)
    if n >= CTA_ROWS - 1:  # two 30 KB values: their tiles exceed the staged byte room and are read from global memory
        vals = s.to_pylist()
        vals[n // 2], vals[n // 4] = LONG_A, LONG_B
        s = pa.array(vals, type=pa.string())
    cols = {
        "s": s,
        "w": _pool_col(rng, [f"w{k:02d}" for k in range(40)], n, pa.string(), 0.03),
        "i": _pool_col(rng, I_POOL, n, pa.int64(), 0.1),
        "f": _pool_col(rng, F_POOL, n, pa.float64(), 0.1),
        "i32": _pool_col(rng, I32_POOL, n, pa.int32(), 0.05),
        "i8": _pool_col(rng, I8_POOL, n, pa.int8(), 0.05),
        "u16": _pool_col(rng, U16_POOL, n, pa.uint16(), 0.05),
        "f32": _pool_col(rng, F32_POOL, n, pa.float32(), 0.05),
        "b": pa.array(rng.random(n) < 0.3, mask=rng.random(n) < 0.1),
        "n": pa.nulls(n, type=pa.string()),
        "hi": pa.array(rng.integers(0, 300_000, n), mask=rng.random(n) < 0.01),
        "a4": pa.array(rng.integers(0, 400, n).astype(np.int32)),
        "b4": pa.array(rng.integers(0, 400, n).astype(np.int32)),
        "t1": pa.array(rng.normal(0, 1, n), mask=rng.random(n) < 0.2),
        "t2": pa.array(rng.integers(-5, 5, n), mask=rng.random(n) < 0.5),
        "tfull": pa.array(rng.normal(0, 1, n)),
        "tnull": pa.nulls(n, type=pa.float64()),
    }
    return pa.table(cols)


# groupings of one plan: (target, group columns); the ids name what runs
SHAPES = {
    "c5_2derived": [("t1", ["s"]), ("t1", ["w"]), ("t1", ["s", "w"])],
    "c5_other_target_0derived": [("t2", ["s"]), ("t2", ["w"]), ("t1", ["s", "w"])],
    "abc_4jobs_3derived": [("t1", ["i", "b", "i32"]), ("t1", ["i"]), ("t1", ["b"]), ("t1", ["i32"])],
    "ab_cd_nc4": [("t1", ["s", "f"]), ("t2", ["i8", "u16"])],
    "five_2batches": [("t1", ["s"]), ("t1", ["w"]), ("t2", ["i"]), ("t2", ["f32"]), ("t1", ["f", "w"])],
    "4col_fallback_only": [("t1", ["s", "w", "i", "f"])],
    "target_is_group": [("s", ["s", "w"]), ("s", ["s"]), ("i", ["i"])],
    "target_no_bitmap": [("tfull", ["s"]), ("tfull", ["w", "i"])],
    "target_all_null": [("tnull", ["s"]), ("tnull", ["s", "w"])],
    "key_all_null": [("t1", ["n"]), ("t1", ["n", "w"])],
    "floats": [("t2", ["f"]), ("t2", ["f32"]), ("t2", ["f", "f32"])],
}
BIG_N = 1_500_003
# at BIG_N every CTA meets > 1024 distinct `hi` values / > 8192 (a4, b4) pairs: the dictionary path overflows into the fallback
BIG_SHAPES = {
    "dict_overflow_fallback": [("t1", ["hi"]), ("t2", ["s"])],
    "comp_overflow_fallback_2derived": [("t1", ["a4", "b4"]), ("t1", ["a4"]), ("t1", ["b4"])],
}
SIZES = [1, CTA_ROWS - 1, CTA_ROWS, CTA_ROWS + 1, 148 * CTA_ROWS - 1, 148 * CTA_ROWS + 1, BIG_N]


def _agg_key(target, groups):
    return "grouped|" + target + "|" + "|".join(groups)


def run_paths(ctx, monkeypatch, name, table, shape, falls_back=False, cache=None, map_limit=50_000):
    """every path setting: exact state and map equal to the reference; launch counts show whether the fallback ran"""
    import term_b200.api as T
    refs = [reference_groups(table, tg, gs, cache=cache) for tg, gs in shape]
    launches, states = {}, {}
    for path in PATHS:
        _set_path(monkeypatch, path)
        plan = T.Plan()
        slots = [T.GroupedCompletenessAnalyzer(tg, gs, max_groups=1 << 21)._add_to(plan) for tg, gs in shape]
        plan.execute_partial(ctx, name)
        launches[path] = plan.stats()["launches"]
        states[path] = []
        for (tg, gs), ref in zip(shape, refs):
            err, msg, got = exact_groups(plan, _agg_key(tg, gs), table, gs)
            assert (err, msg) == (0, ""), (path, tg, gs)
            assert got == ref, (path, tg, gs)
            states[path].append(got)
        plan.finalize()
        for (tg, gs), ref, slot in zip(shape, refs, slots):
            if len(ref) <= map_limit:
                _map_compare(plan.analyzer_result(slot).map, ref, table, gs)
    for path in PATHS:
        assert states[path] == states["default"], path
    # the fingerprint kernel runs one launch + one collection per grouping of a batch; a batch that overflowed the dictionary
    # path paid that many launches before it
    batches = [shape[i: i + 4] for i in range(0, len(shape), 4)]
    extra = sum(1 + len(b) for b in batches) if falls_back else 0
    for path in PATHS:
        if path != "fingerprint":
            assert launches[path] - launches["fingerprint"] == extra, (path, launches)


@pytest.fixture(scope="module")
def tables(ctx):
    made = {}

    def get(n):
        if n not in made:
            t = make_table(n)
            name = f"grp_paths_{n}"
            ctx.register_table(name, t.to_batches(max_chunksize=7001))  # unaligned batches: shifted validity bitmaps
            made[n] = (name, t, {})
        return made[n]

    yield get
    for name, _, _ in made.values():
        ctx.deregister_table(name)


# ------------------------------------------------------------------------------------------------ CPU ----
def _oracle_rendered(table, target, groups):
    def text(x):
        if x is None:
            return b"NULL"
        if isinstance(x, bool):
            return b""
        if isinstance(x, float):
            return O.rust_f64(x).encode()
        if isinstance(x, int):
            return str(x).encode()
        return x.encode()

    return sorted((tuple(text(x) for x in k), t, nn) for k, (t, nn) in O.grouped_completeness(table, target, groups).items())


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_reference_counter_matches_oracle(seed):
    """the reference above against the oracle's GROUP BY on tables where both render every key alike (no ±0.0 / NaN)"""
    rng = np.random.default_rng(seed)
    n = 3000
    u = np.array(["x", "yy", "", "Zeta", "émile", "a longer value than eight", "ab\0"], dtype=object)[rng.integers(0, 7, n)]
    t = pa.table({
        "u": pa.array(u, type=pa.string(), mask=rng.random(n) < 0.1),
        "i": pa.array(rng.integers(-3, 4, n) * 1_000_000_007, mask=rng.random(n) < 0.1),
        "i32": pa.array(rng.integers(-9, 9, n).astype(np.int32), mask=rng.random(n) < 0.05),
        "f": pa.array(rng.integers(1, 6, n) * 0.375 - 4.0, mask=rng.random(n) < 0.1),
        "f32": pa.array((rng.integers(1, 6, n) * 0.25).astype(np.float32)),
        "b": pa.array(rng.random(n) < 0.4, mask=rng.random(n) < 0.1),
        "v": pa.array(rng.normal(0, 1, n), mask=rng.random(n) < 0.3),
    })
    for groups in (["u"], ["i"], ["i32"], ["f"], ["f32"], ["b"], ["u", "i"], ["i32", "f", "b"], ["u", "f32", "i", "b"]):
        assert reference_groups(t, "v", groups) == _oracle_rendered(t, "v", groups), groups
    for c in ("u", "i", "i32", "b"):
        ref = reference_groups(t, c, [c], hist=True)
        buckets = sorted(((f[0], tot) for f, tot, nn in ref if nn), key=lambda e: (-e[1], e[0]))
        h = O.histogram_of(t, c)
        assert [(v.encode(), cnt) for v, cnt, _ in h.buckets] == buckets
        assert sum(tot for f, tot, nn in ref if not nn) == h.null_count


def test_exact_state_parser_on_merged_shards(built_lib):
    """parse_partial / parse_groups on a state the library writes: hand-built shard states (NUL bytes in keys included)
    merged through tg_plan_partial_merge and exported again"""
    import term_b200.api as T
    plan = T.Plan()
    T.GroupedCompletenessAnalyzer("v", ["g"])._add_to(plan)
    (kind, key), = plan.aggregates()
    assert key == _agg_key("v", ["g"])
    groups = [(b"ab", 3, 2), (b"ab\0", 5, 0), (b"", 1, 1), (b"NULL", 4, 4)]

    def shard(entries):
        blob = struct.pack("<Q", len(entries))
        for k, t, nn in entries:
            blob += struct.pack("<I", len(k)) + k + struct.pack("<QQ", t, nn)
        rec = struct.pack("<QQ", kind, 0) + bytes(128) + struct.pack("<Q", len(blob)) + blob + bytes((-len(blob)) % 8) + struct.pack("<Q", 0)
        return struct.pack("<Q", 1) + rec

    plan.partial_reset()
    plan.partial_merge(shard(groups[:2]))
    plan.partial_merge(shard(groups[2:]))
    (_, err, blob, msg), = parse_partial(plan.partial_export())
    assert (err, msg) == (0, "")
    assert sorted(parse_groups(blob)) == sorted(groups)


# ------------------------------------------------------------------------------------------------ GPU ----
@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("n", SIZES)
def test_grouped_paths_match_reference(ctx, tables, monkeypatch, n, shape):
    name, t, cache = tables(n)
    run_paths(ctx, monkeypatch, name, t, SHAPES[shape], cache=cache)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(BIG_SHAPES))
def test_grouped_overflow_falls_back(ctx, tables, monkeypatch, shape):
    name, t, cache = tables(BIG_N)
    run_paths(ctx, monkeypatch, name, t, BIG_SHAPES[shape], falls_back=True, cache=cache)


@pytest.mark.gpu
def test_nine_group_columns_are_refused(ctx, tables, monkeypatch):
    import term_b200.api as T
    name, t, _ = tables(CTA_ROWS + 1)
    gs = ["s", "w", "i", "f", "i32", "i8", "u16", "f32", "b"]
    for path in PATHS:
        _set_path(monkeypatch, path)
        plan = T.Plan()
        ok = T.GroupedCompletenessAnalyzer("t1", ["s"])._add_to(plan)
        bad = T.GroupedCompletenessAnalyzer("t1", gs)._add_to(plan)
        plan.execute_partial(ctx, name)
        assert exact_groups(plan, _agg_key("t1", gs), t, gs)[:2] == (TG_ERR_UNSUPPORTED, "grouped completeness: more than 8 grouping columns")
        plan.finalize()
        r = plan.analyzer_result(bad)
        assert r.error == 2 and r.message == "grouped completeness: more than 8 grouping columns"
        assert plan.analyzer_result(ok).error == 0


@pytest.mark.gpu
def test_targets_sharing_one_validity_buffer(ctx, monkeypatch):
    """two target columns adopted with the SAME validity pointer (the tile kernel stages that bitmap once for both), a
    third with its own; one of the single groupings is derived, the other counted next to it"""
    import torch
    from term_b200 import _ffi as F
    rng = np.random.default_rng(3)
    n = 100_003
    dev = torch.device("cuda", 0)
    g = rng.integers(0, 50, n)
    h = rng.integers(-3, 4, n)
    va, vc = rng.random(n) < 0.7, rng.random(n) < 0.4

    def bitmap(valid):
        b = np.packbits(valid, bitorder="little")
        return torch.from_numpy(np.concatenate([b, np.zeros(64 + (-len(b)) % 64, np.uint8)])).to(dev)

    def values(x, dt):
        return torch.from_numpy(np.concatenate([x.astype(dt), np.zeros(64, dt)])).to(dev)

    tg, th = values(g, np.int64), values(h, np.int64)
    ta, tb, tc = (values(rng.normal(0, 1, n), np.float64) for _ in range(3))
    ba, bc = bitmap(va), bitmap(vc)
    cols = {"g": dict(dtype=F.TG_INT64, n_rows=n, values=tg.data_ptr()), "h": dict(dtype=F.TG_INT64, n_rows=n, values=th.data_ptr()),
            "tA": dict(dtype=F.TG_FLOAT64, n_rows=n, values=ta.data_ptr(), validity=ba.data_ptr()),
            "tB": dict(dtype=F.TG_FLOAT64, n_rows=n, values=tb.data_ptr(), validity=ba.data_ptr()),
            "tC": dict(dtype=F.TG_FLOAT64, n_rows=n, values=tc.data_ptr(), validity=bc.data_ptr())}
    torch.cuda.synchronize()
    ctx.register_device_table("grp_shared_tv", cols, keepalive=[tg, th, ta, tb, tc, ba, bc])
    t = pa.table({"g": pa.array(g), "h": pa.array(h), "tA": pa.array(np.zeros(n), mask=~va), "tB": pa.array(np.zeros(n), mask=~va),
                  "tC": pa.array(np.zeros(n), mask=~vc)})
    try:
        run_paths(ctx, monkeypatch, "grp_shared_tv", t, [("tA", ["g"]), ("tB", ["g"]), ("tB", ["g", "h"]), ("tC", ["h"])])
    finally:
        ctx.deregister_table("grp_shared_tv")


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("n", [40, 700, 2000])
def test_fingerprint_groups_sharing_first_word(ctx, monkeypatch, n, seed):
    """groups whose fingerprints share the first word and differ in the second, in tables one CTA of the fallback kernel
    counts alone: Utf8 values that differ in trailing NUL bytes only, and the Int64 / Float64 value whose bits equal the
    first word of a NULL's pair, next to NULLs"""
    rng = np.random.default_rng(100 * n + seed)
    t = pa.table({
        "s": _pool_col(rng, ["ab", "ab\0", "ab\0\0", "ab\0\0\0"], n, pa.string(), 0.25),
        "i": _pool_col(rng, [NULL_TAG1_I64, 0], n, pa.int64(), 0.4),
        "f": _pool_col(rng, [NULL_TAG1_F64, 1.0], n, pa.float64(), 0.4),
        "v": pa.array(rng.normal(0, 1, n), mask=rng.random(n) < 0.3),
    })
    name = f"grp_race_{n}_{seed}"
    ctx.register_table(name, t)
    try:
        import term_b200.api as T
        _set_path(monkeypatch, "fingerprint")
        for shape in ([("v", ["s"]), ("v", ["i"]), ("v", ["f"]), ("v", ["s", "i"])], [("v", ["i", "f"]), ("v", ["f", "s"])]):
            plan = T.Plan()
            for tg, gs in shape:
                T.GroupedCompletenessAnalyzer(tg, gs)._add_to(plan)
            plan.execute_partial(ctx, name)
            for tg, gs in shape:
                assert exact_groups(plan, _agg_key(tg, gs), t, gs) == (0, "", reference_groups(t, tg, gs)), gs
    finally:
        ctx.deregister_table(name)


def _int_groups(plan, key):
    keys = [k for _, k in plan.aggregates()]
    _, err, blob, msg = parse_partial(plan.partial_export())[keys.index(key)]
    assert (err, msg) == (0, "")
    g = parse_groups(blob)
    k = np.array([int(x) for x, _, _ in g], dtype=np.int64)
    o = np.argsort(k)
    return k[o], np.array([x for _, x, _ in g], dtype=np.int64)[o], np.array([x for _, _, x in g], dtype=np.int64)[o]


@pytest.mark.gpu
def test_exactly_max_groups_are_counted(ctx, monkeypatch):
    import term_b200.api as T
    rng = np.random.default_rng(21)
    n = MAX_GROUPS + 150_001
    keys = rng.permutation(np.concatenate([np.arange(MAX_GROUPS), rng.integers(0, MAX_GROUPS, n - MAX_GROUPS)])) * 7919 - (1 << 40)
    valid = rng.random(n) < 0.75
    t = pa.table({"k": pa.array(keys), "v": pa.array(np.ones(n), mask=~valid)})
    ctx.register_table("grp_limit_ok", t)
    try:
        uniq, inv = np.unique(keys, return_inverse=True)
        tot, nn = np.bincount(inv), np.bincount(inv[valid], minlength=len(uniq))
        assert len(uniq) == MAX_GROUPS
        launches = {}
        for path in ("default", "fingerprint"):
            _set_path(monkeypatch, path)
            plan = T.Plan()
            T.GroupedCompletenessAnalyzer("v", ["k"])._add_to(plan)
            plan.execute_partial(ctx, "grp_limit_ok")
            launches[path] = plan.stats()["launches"]
            gk, gt, gn = _int_groups(plan, _agg_key("v", ["k"]))
            assert np.array_equal(gk, uniq) and np.array_equal(gt, tot) and np.array_equal(gn, nn), path
        assert launches["default"] - launches["fingerprint"] == 2  # the dictionary path overflowed first
    finally:
        ctx.deregister_table("grp_limit_ok")


@pytest.mark.gpu
def test_one_group_over_the_limit_is_refused(ctx, monkeypatch):
    import term_b200.api as T
    n = MAX_GROUPS + 1
    t = pa.table({"k": pa.array(np.random.default_rng(4).permutation(n)), "v": pa.array(np.ones(n))})
    ctx.register_table("grp_limit_over", t)
    try:
        for path in ("default", "fingerprint"):
            _set_path(monkeypatch, path)
            plan = T.Plan()
            slot = T.GroupedCompletenessAnalyzer("v", ["k"])._add_to(plan)
            plan.execute_partial(ctx, "grp_limit_over")
            assert exact_groups(plan, _agg_key("v", ["k"]), t, ["k"])[:2] == (TG_ERR_UNSUPPORTED, LIMIT_MSG)
            plan.finalize()
            r = plan.analyzer_result(slot)
            assert r.error == 2 and r.message == LIMIT_MSG
    finally:
        ctx.deregister_table("grp_limit_over")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["int64", "utf8"])
def test_millions_of_groups_fail_promptly(ctx, monkeypatch, kind):
    """5 M distinct keys overflow every dictionary and exceed the fallback's limit: grouped completeness and the value
    histogram report the limit instead of filling the fallback's global table"""
    import term_b200.api as T
    n = 5_000_000
    keys = pa.array(np.random.default_rng(8).permutation(n))
    if kind == "utf8":
        keys = keys.cast(pa.string())
    t = pa.table({"k": keys, "v": pa.array(np.ones(n), mask=np.arange(n) % 3 == 0)})
    ctx.register_table("grp_5m", t)
    _set_path(monkeypatch, "default")
    try:
        plan = T.Plan()
        slot = T.GroupedCompletenessAnalyzer("v", ["k"])._add_to(plan)
        t0 = time.perf_counter()
        plan.execute(ctx, "grp_5m")
        assert time.perf_counter() - t0 < 30.0
        r = plan.analyzer_result(slot)
        assert r.error == 2 and r.message == LIMIT_MSG
        t0 = time.perf_counter()
        g = T.HistogramConstraint("k", lambda h: True).evaluate(ctx, "grp_5m")
        assert time.perf_counter() - t0 < 30.0
        assert g.status.name == "Failure" and g.message == "Error evaluating constraint: " + LIMIT_MSG
    finally:
        ctx.deregister_table("grp_5m")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["utf8", "int64", "int32", "bool"])
@pytest.mark.parametrize("n", [CTA_ROWS + 1, 120_000])
def test_value_histogram_paths_match_oracle(ctx, monkeypatch, n, kind):
    import term_b200.api as T
    rng = np.random.default_rng(n)
    if kind == "utf8":
        col = _pool_col(rng, [v for v in S_POOL if "\0" not in v] + [LONG_A, LONG_B, "NULL"], n, pa.string(), 0.1)
    elif kind == "int64":
        col = _pool_col(rng, I_POOL, n, pa.int64(), 0.1)
    elif kind == "int32":
        col = _pool_col(rng, I32_POOL + [-7, 9, 10], n, pa.int32(), 0.1)
    else:
        col = pa.array(rng.random(n) < 0.3, mask=rng.random(n) < 0.1)
    t = pa.table({"c": col})
    name = f"hist_paths_{kind}_{n}"
    ctx.register_table(name, t.to_batches(max_chunksize=7001))
    try:
        oh = O.histogram_of(t, "c")
        for path in PATHS:
            _set_path(monkeypatch, path)
            cons = T.HistogramConstraint("c", lambda h: True)
            plan = T.Plan()
            slot = cons._add_to(plan)
            plan.execute(ctx, name)
            h = cons.histogram(plan, slot)
            assert [(b.value, b.count, b.ratio) for b in h.buckets] == oh.buckets, path
            assert (h.total_count, h.null_count, h.distinct_count) == (oh.total_count, oh.null_count, oh.distinct_count), path
    finally:
        ctx.deregister_table(name)
