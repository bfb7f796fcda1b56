"""A failed append leaves the table as it was, on every append path: each test appends valid data, makes a call that fails
part-way (after an earlier column of the batch, the validity bitmap or the column itself has been touched), checks the
status and that the table's row count, column list and every column's buffer record are what they were, then appends
more valid data and compares a suite with the same suite over a table registered from the valid data alone."""
import ctypes as C

import numpy as np
import pyarrow as pa
import pyarrow.parquet as pq
import pytest

import term_b200 as T
from term_b200 import _ffi as F
from tests.test_parquet_bool_int96 import _page

TG_ERR_INVALID_ARG = 1


def _state(ctx, name):
    """(row count, column names in order, per column: dtype, rows, value bytes, NULL count, has a bitmap)"""
    t = C.c_void_p()
    F.check(F.lib().tg_table_lookup(ctx.handle, name.encode(), C.byref(t)))
    d = C.c_int32()
    assert F.lib().tg_table_column_dtype(t, b"no such column", C.byref(d)) == 2  # TG_ERR_COLUMN_NOT_FOUND lists the columns
    listed = F.last_error().split("Valid fields are ", 1)[1][:-1]
    cols = [f.split(".", 1)[1] for f in listed.split(", ")] if listed else []
    bufs = {c: ctx.column_buffers(name, c) for c in cols}
    return ctx.num_rows(name), cols, {c: (b["dtype"], b["n_rows"], b["n_value_bytes"], b["null_count"], bool(b["validity"])) for c, b in bufs.items()}


def _results(ctx, name, value, key):
    A = T.Assertion
    cb = (T.Check.builder("c").has_size(A.GreaterThan(0.0)).has_column_count(A.GreaterThan(0.0)).completeness(value, 0.5).completeness(key, 0.5)
          .has_min(value, A.LessThan(0.0)).has_max(value, A.GreaterThan(0.0)).has_mean(value, A.Between(-1e12, 1e12)))
    res = T.ValidationSuite.builder("s").table_name(name).check(cb.build()).build().run(ctx).report.results
    plan = T.Plan()
    slot = T.GroupedCompletenessAnalyzer(value, [key])._add_to(plan)
    plan.execute(ctx, name)
    return [(r.name, r.status, r.metric, r.message) for r in res], plan.analyzer_result(slot).map


def _same_as_registered(ctx, name, batches, value, key, use_c):
    ctx.register_table("txn_ref", batches, use_c_data_interface=use_c)
    try:
        got, want = _results(ctx, name, value, key), _results(ctx, "txn_ref", value, key)
        assert got == want
    finally:
        ctx.deregister_table("txn_ref")


def _ints(rng, n, null_p):
    return pa.array(rng.integers(-10**9, 10**9, n), mask=rng.random(n) < null_p if null_p else None)


VOCAB = pa.array(["p", "q", "r", "s", "t"])


def _key(kind, rng, n, bad=False):
    """column b: UInt64 below 2^63 (bad: one valid value of 2^63 + 5), or dictionary<int32, utf8> (bad: one valid index
    outside the dictionary)"""
    codes = rng.integers(0, len(VOCAB), n).astype(np.uint64 if kind == "uint64" else np.int32)
    mask = rng.random(n) < 0.1
    if bad:
        codes[n // 2] = 2**63 + 5 if kind == "uint64" else 9
        mask[n // 2] = False
    if kind == "uint64":
        return pa.array(codes, mask=mask)
    return pa.DictionaryArray.from_arrays(pa.array(codes, mask=mask), VOCAB, safe=False)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["uint64", "dictionary"])
def test_failed_record_batch_undoes_its_earlier_columns(ctx, kind):
    rng = np.random.default_rng(11)
    b1 = pa.record_batch([_ints(rng, 1001, 0.0), _key(kind, rng, 1001)], names=["a", "b"])
    # `a` gets its first NULLs (its bitmap is created), `c` is a new column, then `b` is refused
    bad = pa.record_batch([_ints(rng, 777, 0.2), pa.array(rng.random(777)), _key(kind, rng, 777, bad=True)], names=["a", "c", "b"])
    b2 = pa.record_batch([_ints(rng, 503, 0.3), _key(kind, rng, 503)], names=["a", "b"])
    tab = ctx._create("txn_arrow")
    try:
        ctx._append_batch_c(tab, b1)
        before = _state(ctx, "txn_arrow")
        assert not before[2]["a"][4]
        with pytest.raises(F.TermGpuError) as ei:
            ctx._append_batch_c(tab, bad)
        if kind == "uint64":
            assert ei.value.code == F.TG_ERR_UNSUPPORTED and "above the Int64 range" in ei.value.message
        else:
            assert ei.value.code == TG_ERR_INVALID_ARG and "outside the dictionary" in ei.value.message
        assert _state(ctx, "txn_arrow") == before
        ctx._append_batch_c(tab, b2)
        _same_as_registered(ctx, "txn_arrow", [b1, b2], "a", "b", use_c=True)
    finally:
        ctx.deregister_table("txn_arrow")


@pytest.mark.gpu
@pytest.mark.parametrize("had_nulls", [False, True])
def test_failed_utf8_host_append_keeps_null_count_and_bitmap(ctx, had_nulls):
    rng = np.random.default_rng(12)

    def batch(n, null_p):
        words = [f"w{v}" for v in rng.integers(0, 40, n)]
        return pa.record_batch([_ints(rng, n, 0.0), pa.array(words, mask=rng.random(n) < null_p if null_p else None)], names=["x", "s"])
    b1, b2 = batch(1001, 0.2 if had_nulls else 0.0), batch(503, 0.3)
    tab = ctx._create("txn_host")
    try:
        ctx._append_batch(tab, b1, False)
        before = _state(ctx, "txn_host")
        assert before[2]["s"][4] == had_nulls
        # 300 rows with NULLs whose offsets run backwards: refused after the rows' validity has been looked at
        n = 300
        values = np.frombuffer(b"abcdefghij" * 4, dtype=np.uint8)
        offsets = np.linspace(10, 5, n + 1).astype(np.int32)
        validity = np.packbits(rng.random(n) < 0.5, bitorder="little")
        st = F.lib().tg_table_append_host(tab, b"s", F.TG_UTF8, n, values.ctypes.data, offsets.ctypes.data, validity.ctypes.data, 0)
        assert st == TG_ERR_INVALID_ARG and "not monotonic" in F.last_error(), F.last_error()
        assert _state(ctx, "txn_host") == before
        ctx._append_batch(tab, b2, False)
        _same_as_registered(ctx, "txn_host", [b1, b2], "x", "s", use_c=False)
    finally:
        ctx.deregister_table("txn_host")


@pytest.mark.gpu
def test_refused_int96_chunk_leaves_no_column_behind(ctx, tmp_path):
    rng = np.random.default_rng(13)

    def batch(n):
        return pa.record_batch([_ints(rng, n, 0.1), pa.array([f"g{v}" for v in rng.integers(0, 7, n)])], names=["x", "g"])
    b1, b2 = batch(1001), batch(503)
    path = str(tmp_path / "txn.parquet")
    pq.write_table(pa.Table.from_batches([b1]), path)
    ctx.register_parquet("txn_pq", path)
    try:
        before = _state(ctx, "txn_pq")
        tab = C.c_void_p()
        F.check(F.lib().tg_table_lookup(ctx.handle, b"txn_pq", C.byref(tab)))
        chunk = np.frombuffer(_page(b"\x00" * 16, 1001, 5), dtype=np.uint8)  # DELTA_BINARY_PACKED values: refused for INT96
        st = F.lib().tg_table_append_parquet_chunk(tab, b"ts", F.TG_PQ_INT96, 0, 0, chunk.ctypes.data, chunk.size, 1001)
        assert st == F.TG_ERR_UNSUPPORTED and "INT96 values encoded DELTA_BINARY_PACKED" in F.last_error(), F.last_error()
        assert _state(ctx, "txn_pq") == before
        ctx._append_batch_c(tab, b2)
        _same_as_registered(ctx, "txn_pq", [b1, b2], "x", "g", use_c=True)
    finally:
        ctx.deregister_table("txn_pq")
