"""Key-level row verdicts on the GPU (tg_plan_request_key_rows / tg_plan_export_key_rows): DUPLICATE / FIRST of uniqueness
slots and ORPHAN of foreign-key slots, bit-exact against the Counter reference of tests/key_rows_reference.py on every
counting path (single table, dense bitmap, sorted buckets, partitioned buckets, fingerprints), with the popcount identities
checked against the plan's own counts."""
import ctypes as C

import numpy as np
import pyarrow as pa
import pytest

import term_b200 as T
from term_b200 import _ffi as F
from tests import key_rows_reference as KR
from tests.test_row_masks import _read, _register

pytestmark = pytest.mark.gpu
DUP, FIRST, ORPHAN = F.TG_KEY_ROWS_DUPLICATE, F.TG_KEY_ROWS_FIRST, F.TG_KEY_ROWS_ORPHAN
TILE = 4096
BIG = 1_300_000  # above 2^20 rows: the dense / sorted / partitioned paths (conftest lowers their bucket size)
M64 = (1 << 64) - 1


def _fmix64_inv(h):
    h ^= h >> 33
    h = h * 0x9cb4b2f8129337db & M64
    h ^= h >> 33
    h = h * 0x4f74430c22a54005 & M64
    h ^= h >> 33
    return h - (1 << 64) if h >= 1 << 63 else h


SORTED_SPECIAL = _fmix64_inv(M64)  # the key the sorted-bucket path counts apart (its hash is the table's EMPTY word)


def _strs(*a):
    return (C.c_char_p * len(a))(*[s.encode() for s in a])


def _uniq_plan(columns, request=True):
    p = T.api.Plan()
    lib, A = F.lib(), F.tg_assertion(0, 0.0, 0.0)
    full = lib.tg_plan_add_uniqueness(p.handle, _strs(*columns), len(columns), 0, 1.0, A, 0)
    ratio = lib.tg_plan_add_uniqueness(p.handle, _strs(*columns), len(columns), 2, 0.0, A, 0)
    pk = lib.tg_plan_add_uniqueness(p.handle, _strs(*columns), len(columns), 3, 0.0, A, 0)
    if request:
        p.request_key_rows(full, DUP)
        p.request_key_rows(pk, FIRST)
    return p, full, ratio, pk


def _check_uniqueness(ctx, table, columns):
    _register(ctx, "kr_data", table)
    p, full, ratio, pk = _uniq_plan(columns)
    p.execute(ctx, "kr_data")
    n = table.num_rows
    dup, dup_ok = _read(p.key_rows(full, DUP))
    first, first_ok = _read(p.key_rows(pk, FIRST))
    want_dup, want_first, want_ok = (np.array(x, dtype=bool) for x in KR.uniqueness_rows(table, columns))
    assert np.array_equal(dup_ok, want_ok) and np.array_equal(first_ok, want_ok)
    assert np.array_equal(dup & dup_ok, want_dup), np.flatnonzero((dup & dup_ok) != want_dup)[:10]
    assert np.array_equal(first & first_ok, want_first), np.flatnonzero((first & first_ok) != want_first)[:10]
    if n == 0:
        return
    # the plan's own counts: FULL = COUNT(DISTINCT ..) / rows, UNIQUE_VALUE_RATIO = singleton groups / rows
    single, nulls = len(columns) == 1, n - int(want_ok.sum())
    assert int((first & first_ok).sum()) == round(p.result(full).metric * n)
    singles = round(p.result(ratio).metric * n) - (1 if single and nulls == 1 else 0)
    assert int((dup & dup_ok).sum()) == int(want_ok.sum()) - singles
    return p


def _ints(rng, n, null_p, pool):
    keys = rng.choice(np.asarray(pool, dtype=np.int64), n)
    mask = None if null_p == 0 else (np.ones(n, bool) if null_p == 1.0 else rng.random(n) < null_p)
    return pa.array(keys, type=pa.int64(), mask=mask)


@pytest.mark.parametrize("n", [0, 1, 31, 32, 33, TILE - 1, TILE + 5])
@pytest.mark.parametrize("null_p", [0.0, 0.05, 1.0])
def test_single_table_int64_and_float64(ctx, n, null_p):
    rng = np.random.default_rng(n * 7 + int(null_p * 100))
    a = _ints(rng, n, null_p, [-1, 0, 5, 7, 1 << 40, -(1 << 62)] + list(range(100, 100 + n)))
    fv = rng.choice(np.array([0.0, -0.0, np.nan, -np.nan, 1.5, -2.25, np.inf]), n)
    f = pa.array(fv, mask=None if null_p == 0 else rng.random(n) < null_p)
    t = pa.table({"a": a, "f": f})
    _check_uniqueness(ctx, t, ["a"])
    _check_uniqueness(ctx, t, ["f"])


@pytest.mark.parametrize("n", [31, 33, TILE + 5, 70_000])
@pytest.mark.parametrize("null_p", [0.0, 0.05, 1.0])
def test_fingerprint_keys(ctx, n, null_p):
    rng = np.random.default_rng(n + int(null_p * 10))
    words = np.array(["", "a", "ab", "héllo", "日本", "x" * 40] + [f"k{i}" for i in range(n // 2)], dtype=object)
    mask = None if null_p == 0 else (np.ones(n, bool) if null_p == 1.0 else rng.random(n) < null_p)
    t = pa.table({"s": pa.array(list(rng.choice(words, n)), type=pa.string(), mask=mask),
                  "a": _ints(rng, n, null_p / 2, [-1, 0, 1, 2]),
                  "i": pa.array(rng.integers(0, 3, n).astype(np.int32))})
    _check_uniqueness(ctx, t, ["s"])
    _check_uniqueness(ctx, t, ["i"])
    _check_uniqueness(ctx, t, ["a", "s"])


def _big_sparse(rng, n, null_p=0.05):
    pool = rng.integers(-(1 << 62), 1 << 62, n // 2)
    pool[:3] = [-1, SORTED_SPECIAL, 0]
    keys = rng.choice(pool, n)
    keys[:4] = [-1, -1, SORTED_SPECIAL, SORTED_SPECIAL]  # both sentinel keys, repeated
    return pa.array(keys, mask=rng.random(n) < null_p)


@pytest.mark.parametrize("path", ["dense", "sorted", "sorted_f64", "partitioned", "hot_key"])
def test_large_paths(ctx, monkeypatch, path):
    rng = np.random.default_rng(11)
    if path == "dense":
        a = pa.array(rng.integers(-1, 700_000, BIG), mask=rng.random(BIG) < 0.05)
    elif path == "sorted_f64":
        a = pa.array(np.where(rng.random(BIG) < 0.01, -0.0, rng.integers(0, 600_000, BIG) * 0.5), mask=rng.random(BIG) < 0.05)
        v = a.to_numpy(zero_copy_only=False)
        v[:6] = [0.0, -0.0, np.nan, -np.nan, np.nan, 1.0]
        a = pa.array(v, mask=rng.random(BIG) < 0.05)
    elif path == "hot_key":  # sorted buckets give up on a key with more copies than a bucket: partitioned
        v = rng.integers(-(1 << 62), 1 << 62, BIG)
        v[rng.random(BIG) < 0.35] = 123456789
        a = pa.array(v)
    else:
        a = _big_sparse(rng, BIG)
    if path == "partitioned":
        monkeypatch.setenv("TG_HASH_NO_SORTED", "1")
    _check_uniqueness(ctx, pa.table({"a": a}), ["a"])


@pytest.mark.parametrize("kind", ["dense", "sorted", "partitioned", "utf8"])
def test_repeated_key_table_redo(ctx, monkeypatch, kind):
    """more repeated keys (2^20 + 75 K) than the first R (2^20 slots) has places for: the first pass stops inserting at half,
    the job is repeated once with R sized from the count, and the hash job's device time stays that of two counting passes"""
    rng = np.random.default_rng(5)
    keys = np.concatenate([np.arange(1_123_000), np.arange(1_123_000)]) * (1 if kind == "dense" else 7919)
    rng.shuffle(keys)
    if kind == "sorted":
        monkeypatch.setenv("TG_HASH_NO_DENSE", "1")
    if kind == "partitioned":
        monkeypatch.setenv("TG_HASH_NO_DENSE", "1")
        monkeypatch.setenv("TG_HASH_NO_SORTED", "1")
    col = pa.array([f"s{x}" for x in keys], type=pa.string()) if kind == "utf8" else pa.array(keys)
    p = _check_uniqueness(ctx, pa.table({"a": col}), ["a"])
    print(f"{kind}: hash job {p.stats()['hash_ms']:.2f} ms device time")
    assert p.stats()["hash_ms"] < 1000.0


def test_results_unchanged_by_requests(ctx):
    rng = np.random.default_rng(2)
    for t in (pa.table({"a": _big_sparse(rng, BIG)}), pa.table({"a": _ints(rng, 5000, 0.05, list(range(-1, 3000)))})):
        _register(ctx, "kr_data", t)
        a = _uniq_plan(["a"], request=True)
        b = _uniq_plan(["a"], request=False)
        a[0].execute(ctx, "kr_data")
        b[0].execute(ctx, "kr_data")
        for sa, sb in zip(a[1:], b[1:]):
            ra, rb = a[0].result(sa), b[0].result(sb)
            assert (ra.status, ra.metric, ra.message) == (rb.status, rb.metric, rb.message)
    # FULL alone on a dense column: unrequested, the bitmap path counts with non-returning ORs (no singleton count); a
    # request switches it to the seen-twice mode
    _register(ctx, "kr_data", pa.table({"a": pa.array(rng.integers(0, 900_000, BIG), mask=rng.random(BIG) < 0.05)}))
    lib, A, res = F.lib(), F.tg_assertion(0, 0.0, 0.0), []
    for request in (True, False):
        p = T.api.Plan()
        s = lib.tg_plan_add_uniqueness(p.handle, _strs("a"), 1, 0, 1.0, A, 0)
        if request:
            p.request_key_rows(s, FIRST)
        p.execute(ctx, "kr_data")
        r = p.result(s)
        res.append((r.status, r.metric, r.message))
    assert res[0] == res[1]


# ------------------------------------------------------------------------------------------ foreign keys ----
def _check_fk(ctx, child, parent, allow_nulls, request=True):
    _register(ctx, "kr_child", pa.table({"c": child}))
    _register(ctx, "kr_parent", pa.table({"p": parent}))
    p = T.api.Plan()
    s = F.lib().tg_plan_add_foreign_key(p.handle, b"kr_child.c", b"kr_parent.p", allow_nulls, 10)
    q = T.api.Plan()
    s2 = F.lib().tg_plan_add_foreign_key(q.handle, b"kr_child.c", b"kr_parent.p", allow_nulls, 10)
    p.request_key_rows(s, ORPHAN)
    p.execute(ctx, "kr_child")
    q.execute(ctx, "kr_child")
    r, r2 = p.result(s), q.result(s2)
    # unchanged by the request (the examples are an unordered DISTINCT .. LIMIT: which ones is not pinned)
    assert (r.status, r.metric, (r.message or "").split(" Examples:")[0]) == (r2.status, r2.metric, (r2.message or "").split(" Examples:")[0])
    m = p.key_rows(s, ORPHAN)
    assert m.length == len(child)
    vals, valid = _read(m)
    tables = {"kr_child": pa.table({"c": child}), "kr_parent": pa.table({"p": parent})}
    want, want_ok = (np.array(x, dtype=bool) for x in KR.orphan_rows(tables, "kr_child.c", "kr_parent.p"))
    assert np.array_equal(valid, want_ok)
    assert np.array_equal(vals & valid, want), np.flatnonzero((vals & valid) != want)[:10]
    nulls = len(child) - int(want_ok.sum())
    assert m.null_count == nulls
    violations = 0 if r.metric is None else round(r.metric)
    assert int((vals & valid).sum()) == violations - (0 if allow_nulls else nulls)


@pytest.mark.parametrize("allow_nulls", [0, 1])
@pytest.mark.parametrize("path", ["single", "single_parent_minus1", "single_sparse", "single_f64", "dense", "partitioned",
                                  "partitioned_parent_minus1", "utf8", "empty_parent", "empty_parent_utf8", "no_orphan", "empty_child"])
def test_foreign_key_paths(ctx, path, allow_nulls):
    # single*: at most 2^20 child rows and a parent below the bucket size (conftest: 262144 keys) take the single-table probe
    # (fk_probe64_kernel's collect pass), whatever the parent's range; Float64 keys always do
    rng = np.random.default_rng(len(path) + allow_nulls)
    if path == "single_sparse":
        parent = rng.integers(-(1 << 62), 1 << 62, 1000)
        child = np.where(rng.random(5000) < 0.5, rng.choice(parent, 5000), rng.integers(-(1 << 62), 1 << 62, 5000))
        child[:3] = -1
    elif path == "single_f64":
        pool = np.array([0.0, -0.0, 1.5, -1.0, np.nan, np.inf, 2.0 ** 60, -3.25])
        parent = pa.array(np.array([0.0, 1.5, np.inf, 7.0]))
        child = rng.choice(pool, 5000)
        _check_fk(ctx, pa.array(child, mask=rng.random(5000) < 0.05), parent, allow_nulls)
        return
    elif path.startswith("single"):
        parent = np.arange(0, 2000, 2)
        child = rng.integers(-1, 3000, 5000)
        if path.endswith("minus1"):
            parent = np.append(parent, -1)
    elif path == "dense":  # dense Int64 parent range: a bitmap
        parent = np.arange(0, 400_000)
        child = rng.integers(-1, 500_000, BIG)
    elif path.startswith("partitioned"):  # a sparse parent too large for one L2 table: partitioned buckets
        parent = rng.integers(-(1 << 62), 1 << 62, 300_000)
        child = np.where(rng.random(400_000) < 0.5, rng.choice(parent, 400_000), rng.integers(-(1 << 62), 1 << 62, 400_000))
        child[:5] = -1
        if path.endswith("minus1"):
            parent[7] = -1
    elif path == "utf8":
        parent = pa.array([f"p{i}" for i in range(3000)] + [None])
        child = pa.array([f"p{i}" if i % 3 else f"q{i % 500}" for i in rng.integers(0, 4000, 20_000)],
                         mask=rng.random(20_000) < 0.05)
        _check_fk(ctx, child, parent, allow_nulls)
        return
    elif path == "empty_parent_utf8":
        _check_fk(ctx, pa.array(["a", None, "b", "a"]), pa.array([], type=pa.string()), allow_nulls)
        return
    elif path == "empty_parent":
        parent = np.array([], dtype=np.int64)
        child = rng.integers(-1, 10, 100)
    elif path == "empty_child":
        _check_fk(ctx, pa.array([], type=pa.int64()), pa.array([1, 2]), allow_nulls)
        return
    else:  # no key violates: only the NULL children can
        parent = np.arange(-1, 1000)
        child = rng.integers(-1, 1000, 3000)
    _check_fk(ctx, pa.array(child, mask=rng.random(len(child)) < 0.05), pa.array(parent, type=pa.int64()), allow_nulls)


@pytest.mark.parametrize("path", ["dense", "partitioned"])
def test_orphan_table_redo(ctx, path):
    """more than 2^19 distinct orphans: the paths repeat their probe with an exact-size table"""
    rng = np.random.default_rng(8)
    if path == "dense":
        parent = np.arange(0, 400_000)
        child = np.concatenate([rng.integers(0, 400_000, 500_000), np.arange(1_000_000, 1_700_000)])
    else:
        parent = rng.integers(-(1 << 62), 1 << 62, 300_000)
        child = np.concatenate([rng.choice(parent, 100_000), rng.integers(-(1 << 62), 1 << 62, 700_000)])
    rng.shuffle(child)
    _check_fk(ctx, pa.array(child, mask=rng.random(len(child)) < 0.01), pa.array(parent), 0)


# ---------------------------------------------------------------------------------------- lifetime, shards ----
def test_lifetime_after_reexecute_and_destroy(ctx):
    rng = np.random.default_rng(4)
    t = pa.table({"a": _ints(rng, 3000, 0.05, list(range(-1, 1000)))})
    _register(ctx, "kr_data", t)
    p, full, _, pk = _uniq_plan(["a"])
    p.execute(ctx, "kr_data")
    old = p.key_rows(full, DUP)
    old_bits = _read(old)
    h = C.c_void_p()
    F.check(F.lib().tg_table_lookup(ctx.handle, b"kr_data", C.byref(h)))
    for b in pa.table({"a": _ints(rng, 500, 0.05, list(range(-1, 1000)))}).to_batches():
        ctx._append_batch(h, b, False)
    p.execute(ctx, "kr_data")
    new = p.key_rows(full, DUP)
    assert new.length == 3500 and old.length == 3000
    assert all(np.array_equal(x, y) for x, y in zip(_read(old), old_bits))
    p.request_key_rows(full, FIRST)  # a request after the last execute: unavailable until the next one
    with pytest.raises(T.TermGpuError):
        p.key_rows(full, FIRST)
    del p
    import gc
    gc.collect()
    assert all(np.array_equal(x, y) for x, y in zip(_read(old), old_bits))  # survives the plan


def test_shuffled_keys_are_refused(ctx):
    rng = np.random.default_rng(6)
    t = pa.table({"a": _ints(rng, 1000, 0.0, list(range(100)))})
    _register(ctx, "kr_data", t)
    _register(ctx, "kr_shard", t.slice(0, 400))
    p, full, _, _ = _uniq_plan(["a"])
    F.check(F.lib().tg_plan_redirect_aggregate(p.handle, 0, 0, b"kr_shard"))
    p.execute(ctx, "kr_data")
    assert p.result(full).metric is not None
    with pytest.raises(T.TermGpuError) as e:
        p.key_rows(full, DUP)
    assert e.value.code == F.TG_ERR_UNSUPPORTED and "shuffled" in str(e.value)
    _register(ctx, "kr_child", pa.table({"c": pa.array([1, 2, 3])}))
    _register(ctx, "kr_parent", pa.table({"p": pa.array([1])}))
    q = T.api.Plan()
    s = F.lib().tg_plan_add_foreign_key(q.handle, b"kr_child.c", b"kr_parent.p", 0, 10)
    q.request_key_rows(s, ORPHAN)
    F.check(F.lib().tg_plan_redirect_aggregate(q.handle, 0, 1, b"kr_parent"))
    q.execute(ctx, "kr_child")
    with pytest.raises(T.TermGpuError) as e:
        q.key_rows(s, ORPHAN)
    assert e.value.code == F.TG_ERR_UNSUPPORTED


def test_125m_keys_against_torch(ctx):
    import torch
    from term_b200.distributed import _tensor_from_ptr
    n = 125_000_000
    rng = np.random.default_rng(1)
    keys = rng.integers(0, 100_000_000, n)
    _register(ctx, "kr_big", pa.table({"a": keys}))
    p, full, _, pk = _uniq_plan(["a"])
    p.execute(ctx, "kr_big")  # about 35 M repeated keys: the first R stops at half and the job is repeated once
    print(f"125 M keys: hash job {p.stats()['hash_ms']:.2f} ms device time")
    assert p.stats()["hash_ms"] < 1000.0
    dev = torch.device("cuda", 0)
    k = torch.from_numpy(keys).to(dev)
    del keys
    uniq, inv, counts = torch.unique(k, return_inverse=True, return_counts=True)
    rows = torch.arange(n, device=dev)
    first_row = torch.full((uniq.numel(),), n, device=dev, dtype=torch.int64).scatter_reduce(0, inv, rows, "amin")
    want_dup, want_first = counts[inv] >= 2, first_row[inv] == rows
    shifts = torch.arange(8, device=dev, dtype=torch.uint8)

    def bits(m):
        raw = _tensor_from_ptr(m.values_ptr, (n + 7) // 8, dev, "|u1")[: (n + 7) // 8]
        return ((raw.unsqueeze(1) >> shifts) & 1).reshape(-1)[:n].bool()

    d, f = p.key_rows(full, DUP), p.key_rows(pk, FIRST)
    assert d.validity_ptr == 0 and d.null_count == 0
    assert torch.equal(bits(d), want_dup)
    assert torch.equal(bits(f), want_first)
    assert int(want_first.sum()) == uniq.numel() == round(p.result(full).metric * n)
