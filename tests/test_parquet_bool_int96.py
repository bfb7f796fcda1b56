"""Parquet BOOLEAN and INT96 column chunks -> HBM. BOOLEAN chunks (PLAIN in V1 data pages, RLE in V2 data pages as pyarrow
writes them) become the bit-packed Arrow Boolean values; INT96 chunks (the legacy Impala / Hive / Spark timestamp,
dictionary-encoded by default) become Int64 nanoseconds since the epoch, delivered as Timestamp(Nanosecond, None). Files
are written here with pyarrow and its reader is the ground truth. CPU tests: the host page walk, the validity bitmap and
the Python type mapping. GPU tests: the decoded buffers bit for bit, appends at unaligned rows, a suite against the same
suite over pyarrow's read of the file, malformed and refused chunks, and a 100 M-row Boolean column."""
import os

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc
import pyarrow.parquet as pq
import pytest

import term_b200 as T
from term_b200 import _ffi as F

# (rows, NULL fraction, row-group size, dictionary page limit of the INT96 column: small -> PLAIN fallback part-way)
CASES = [(1, 0.0, None, None), (1000, 0.3, None, None), (300_000, 0.05, 100_000, 4096), (70_001, 1.0, None, None),
         (200_000, 0.999, None, None), (50_000, 0.0, None, 2048)]


def _table(n, null_p, seed):
    rng = np.random.default_rng(seed + n)
    days = rng.integers(-20_000, 30_000, n)  # 1915 .. 2052
    ts = days * 86_400 * 10**9 + rng.integers(0, 86_400 * 10**9, n)
    return pa.table({
        "b": pa.array(rng.random(n) < 0.4, mask=rng.random(n) < null_p),
        "runs": pa.array(np.sort(rng.random(n)) < 0.7, mask=rng.random(n) < null_p),   # long runs
        "breq": pa.array(rng.random(n) < 0.5),
        "ts": pa.array(ts, type=pa.timestamp("ns"), mask=rng.random(n) < null_p),
        "tsc": pa.array(rng.integers(0, 40, n) * 3_600 * 10**9 + 10**18, type=pa.timestamp("ns")),  # few distinct instants
        "x": pa.array(rng.normal(0, 1, n), mask=rng.random(n) < null_p),
    }, schema=pa.schema([pa.field("b", pa.bool_()), pa.field("runs", pa.bool_()), pa.field("breq", pa.bool_(), nullable=False),
                         pa.field("ts", pa.timestamp("ns")), pa.field("tsc", pa.timestamp("ns"), nullable=False), pa.field("x", pa.float64())]))


def _write(tmp_path, n, null_p, row_group, version, compression="NONE", dict_limit=None, seed=1, page=16 * 1024):
    t = _table(n, null_p, seed)
    path = os.path.join(str(tmp_path), f"bi_{n}_{version}_{compression}_{seed}.parquet")
    kw = dict(dictionary_pagesize_limit=dict_limit) if dict_limit else {}
    pq.write_table(t, path, compression=compression, data_page_version=version, row_group_size=row_group, data_page_size=page,
                   use_deprecated_int96_timestamps=True, **kw)
    return path, t


def _chunks(path):
    """(column name, chunk bytes as ndarray, column metadata, leaf) for every column chunk of the file"""
    pf = pq.ParquetFile(path)
    md, raw = pf.metadata, open(path, "rb").read()
    for rg in range(md.num_row_groups):
        for ci in range(md.num_columns):
            cm = md.row_group(rg).column(ci)
            start = cm.dictionary_page_offset if cm.has_dictionary_page and cm.dictionary_page_offset else cm.data_page_offset
            yield rg, cm.path_in_schema, np.frombuffer(raw[start: start + cm.total_compressed_size], dtype=np.uint8), cm, pf.schema.column(ci)


# ------------------------------------------------------------------------------------------ CPU ----
@pytest.mark.parametrize("compression", ["NONE", "SNAPPY"])
@pytest.mark.parametrize("version", ["1.0", "2.0"])
@pytest.mark.parametrize("n,null_p,row_group,dict_limit", CASES)
def test_page_walk_and_validity_of_boolean_and_int96_chunks(built_lib, tmp_path, n, null_p, row_group, dict_limit, version, compression):
    path, t = _write(tmp_path, n, null_p, row_group, version, compression, dict_limit)
    md = pq.ParquetFile(path).metadata
    row0 = {}
    for rg, name, chunk, cm, leaf in _chunks(path):
        if name == "x":
            continue
        n_pages = F.lib().tg_parquet_inspect_chunk(chunk.ctypes.data, chunk.size, None, 0)
        assert n_pages > 0, F.last_error()
        pages = (F.tg_parquet_page * n_pages)()
        assert F.lib().tg_parquet_inspect_chunk(chunk.ctypes.data, chunk.size, pages, n_pages) == n_pages
        data = [p for p in pages if p.page_type in (0, 3)]
        assert sum(p.num_values for p in data) == cm.num_values
        assert all(p.page_type == (0 if version == "1.0" else 3) for p in data)
        if cm.physical_type == "BOOLEAN":
            assert all(p.page_type != 2 for p in pages)
            assert all(p.encoding == (0 if version == "1.0" else 3) for p in data), [p.encoding for p in data]  # PLAIN (V1) / RLE (V2)
        else:
            assert cm.physical_type == "INT96"
            assert pages[0].page_type == 2 and pages[0].encoding in (0, 2) and all(p.encoding in (0, 2, 8) for p in data)
            if dict_limit and name == "ts" and n > 10_000:
                assert any(p.encoding == 0 for p in data), "no PLAIN fallback"
        if leaf.max_definition_level and (compression == "NONE" or version == "2.0"):  # (the validity walk does not inflate V1 pages)
            r0 = row0.get(name, 0)
            bits = np.zeros((cm.num_values + 7) // 8, dtype=np.uint8)
            nn = F.lib().tg_parquet_chunk_validity(chunk.ctypes.data, chunk.size, cm.num_values, bits.ctypes.data)
            want = np.asarray(t.column(name).slice(r0, cm.num_values).is_valid())
            got = np.unpackbits(bits, bitorder="little")[: cm.num_values].astype(bool)
            assert nn == int(want.sum()) and (got == want).all(), (name, rg)
        row0[name] = row0.get(name, 0) + cm.num_values
    assert md.num_rows == n


def test_boolean_and_int96_map_to_device_types(built_lib, tmp_path):
    S = T.SessionContext
    assert S._PARQUET_TYPES["BOOLEAN"] == F.TG_BOOL and S._PARQUET_TYPES["INT96"] == F.TG_PQ_INT96 == 8
    path, _ = _write(tmp_path, 10, 0.0, None, "1.0")
    schema = pq.ParquetFile(path).schema
    for i in range(len(schema)):
        leaf = schema.column(i)
        assert S._check_parquet_logical_type(leaf.name, leaf) is None, leaf.name   # the engine declares INT96 itself


# ------------------------------------------------------------------------------------------ GPU ----
def _read(ctx, table, column):
    """(raw value bytes, validity bool ndarray, buffers) of a device column"""
    import torch
    from term_b200.distributed import _tensor_from_ptr
    b = ctx.column_buffers(table, column)
    dev = torch.device("cuda", 0)
    n = b["n_rows"]
    nbytes = (n + 7) // 8 if b["dtype"] == F.TG_BOOL else n * 8
    vals = _tensor_from_ptr(b["values"], max(nbytes, 1), dev, "|u1").cpu().numpy()[:nbytes]
    if b["validity"]:
        bits = _tensor_from_ptr(b["validity"], (n + 7) // 8, dev, "|u1").cpu().numpy()
        valid = np.unpackbits(bits, bitorder="little")[:n].astype(bool)
    else:
        valid = np.ones(n, dtype=bool)
    return vals, valid, b


def _check_bool(ctx, table, column, want, nulls_read_zero=True):
    """value bits of valid rows, validity, NULL rows read 0 (rows appended from Arrow keep the bits they came with), the
    bits past the last row are 0"""
    vals, valid, b = _read(ctx, table, column)
    want = want.combine_chunks() if isinstance(want, pa.ChunkedArray) else want
    n = len(want)
    assert b["n_rows"] == n and b["dtype"] == F.TG_BOOL and b["n_value_bytes"] == (n + 7) // 8
    want_valid = np.asarray(want.is_valid())
    assert (valid == want_valid).all(), column
    assert b["null_count"] == int((~want_valid).sum())
    got = np.unpackbits(vals, bitorder="little")
    want_bits = np.asarray(want.fill_null(False)).astype(np.uint8)
    keep = np.ones(n, dtype=bool) if nulls_read_zero else want_valid
    assert (got[:n][keep] == want_bits[keep]).all(), (column, np.flatnonzero((got[:n] != want_bits) & keep)[:10])
    assert not got[n:].any(), column


def _check_ts(ctx, table, column, want):
    vals, valid, b = _read(ctx, table, column)
    want = want.combine_chunks() if isinstance(want, pa.ChunkedArray) else want
    n = len(want)
    assert b["n_rows"] == n and b["dtype"] == F.TG_INT64
    want_valid = np.asarray(want.is_valid())
    assert (valid == want_valid).all(), column
    got = vals.view(np.int64)
    w = np.asarray(want.cast(pa.int64()).fill_null(0))
    assert (got[want_valid] == w[want_valid]).all(), column
    assert (got[~want_valid] == 0).all(), column


@pytest.mark.gpu
@pytest.mark.parametrize("compression", ["NONE", "SNAPPY", "ZSTD"])
@pytest.mark.parametrize("version", ["1.0", "2.0"])
@pytest.mark.parametrize("n,null_p,row_group,dict_limit", CASES)
def test_boolean_and_int96_chunks_decode_to_the_arrow_layout(ctx, tmp_path, n, null_p, row_group, dict_limit, version, compression):
    path, _ = _write(tmp_path, n, null_p, row_group, version, compression, dict_limit, page=4 * 1024)  # many small pages
    want = pq.read_table(path)
    assert want.schema.field("ts").type == pa.timestamp("ns")
    name = "pqbi"
    ctx.register_parquet(name, path)
    try:
        assert ctx.num_rows(name) == n
        for col in ("b", "runs", "breq"):
            _check_bool(ctx, name, col, want.column(col))
        for col in ("ts", "tsc"):
            _check_ts(ctx, name, col, want.column(col))
    finally:
        ctx.deregister_table(name)


# ---- hand-built pages: run structures pyarrow's writer never emits ----
def _varint(v):
    out = bytearray()
    while True:
        b = v & 0x7F
        v >>= 7
        out.append(b | (0x80 if v else 0))
        if not v:
            return bytes(out)


def _zz(v):
    return _varint((v << 1) ^ (v >> 63))


def _page(values: bytes, num_values: int, encoding: int, levels: bytes = None, page_type: int = 0) -> bytes:
    """a V1 data page (levels: the RLE definition levels of an optional column, None: a required column) or, with
    page_type 2, a dictionary page"""
    body = (len(levels).to_bytes(4, "little") + levels if levels is not None else b"") + values
    if page_type == 2:  # DictionaryPageHeader {1 num_values, 2 encoding}: field id 7
        return b"\x15" + _zz(2) + b"\x15" + _zz(len(body)) + b"\x15" + _zz(len(body)) + b"\x7c" + b"\x15" + _zz(num_values) + b"\x15" + _zz(encoding) + b"\x00\x00" + body
    dph = b"\x15" + _zz(num_values) + b"\x15" + _zz(encoding) + b"\x15" + _zz(3) + b"\x15" + _zz(3) + b"\x00"
    return b"\x15" + _zz(0) + b"\x15" + _zz(len(body)) + b"\x15" + _zz(len(body)) + b"\x2c" + dph + b"\x00" + body


def _hybrid(runs):
    """runs: ("rle", count, bit) | ("packed", [bits...]); only the stream's last packed run may end in a padded group"""
    out, bits = bytearray(), []
    for r in runs:
        if r[0] == "rle":
            out += _varint(r[1] << 1) + bytes([r[2]])
            bits += [r[2]] * r[1]
        else:
            b = list(r[1])
            groups = (len(b) + 7) // 8
            out += _varint((groups << 1) | 1) + np.packbits(np.array(b + [0] * (groups * 8 - len(b)), dtype=np.uint8), bitorder="little").tobytes()
            bits += b
    return bytes(out), np.array(bits, dtype=bool)


def _rle_values(runs):
    stream, bits = _hybrid(runs)
    return len(stream).to_bytes(4, "little") + stream, bits


def _random_runs(rng, k_max=40):
    runs = []
    for _ in range(int(rng.integers(1, k_max))):
        if rng.random() < 0.5:
            runs.append(("rle", int(rng.choice([1, 7, 8, 9, 31, 32, 33, 1023, 1024, 1025, 5000])), int(rng.integers(0, 2))))
        else:
            runs.append(("packed", rng.integers(0, 2, 8 * int(rng.integers(1, 200))).tolist()))
    runs.append(("packed", rng.integers(0, 2, int(rng.integers(1, 8))).tolist()))  # padded last group
    return runs


def _append_chunk(tab, col, dtype, max_def, chunk_bytes, n):
    chunk = np.frombuffer(chunk_bytes, dtype=np.uint8)
    return F.lib().tg_table_append_parquet_chunk(tab, col.encode(), dtype, max_def, 0, chunk.ctypes.data, chunk.size, n)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(8))
def test_hand_built_boolean_pages_decode_exactly(ctx, seed):
    """RLE pages with long runs, runs across 1024-row blocks, padded last groups and single-value pages, mixed with PLAIN
    pages, required and optional (the RLE stream then holds only the non-NULL values)"""
    rng = np.random.default_rng(seed)
    for optional in (False, True):
        pages, vals_all, valid_all = [], [], []
        for p in range(int(rng.integers(1, 6))):
            if p == 0 and seed % 2:
                n_rows = 1  # a single-value page
            else:
                n_rows = int(rng.integers(1, 9000))
            valid = rng.random(n_rows) < 0.7 if optional else np.ones(n_rows, dtype=bool)
            nn = int(valid.sum())
            if rng.random() < 0.7:
                runs = _random_runs(rng)
                _, bits = _hybrid(runs)
                while len(bits) < nn:  # cover every non-NULL row
                    runs = runs[:-1] + [("rle", nn - len(bits) + 3, int(rng.integers(0, 2)))] + runs[-1:]
                    _, bits = _hybrid(runs)
                values, bits = _rle_values(runs)
                enc = 3
            else:
                bits = rng.random(nn) < 0.5
                values = np.packbits(bits.astype(np.uint8), bitorder="little").tobytes()
                enc = 0
            levels = _hybrid([("packed", valid.astype(int).tolist())])[0] if optional else None
            pages.append(_page(values, n_rows, enc, levels))
            v = np.zeros(n_rows, dtype=bool)
            v[valid] = bits[:nn]
            vals_all.append(v)
            valid_all.append(valid)
        want = pa.array(np.concatenate(vals_all), mask=~np.concatenate(valid_all))
        tab = ctx._create("hb")
        try:
            F.check(_append_chunk(tab, "b", F.TG_BOOL, int(optional), b"".join(pages), len(want)))
            _check_bool(ctx, "hb", "b", want)
        finally:
            ctx.deregister_table("hb")


@pytest.mark.gpu
def test_two_files_appended_at_an_unaligned_row(ctx, tmp_path):
    p1, t1 = _write(tmp_path, 70_001, 0.3, None, "2.0", "SNAPPY", seed=3)
    p2, t2 = _write(tmp_path, 300_000, 0.05, 100_000, "1.0", "ZSTD", 4096, seed=4)
    ctx.register_parquet("pqa", [p1, p2])
    try:
        want = pa.concat_tables([pq.read_table(p1), pq.read_table(p2)])
        for col in ("b", "runs", "breq"):
            _check_bool(ctx, "pqa", col, want.column(col))
        for col in ("ts", "tsc"):
            _check_ts(ctx, "pqa", col, want.column(col))
    finally:
        ctx.deregister_table("pqa")


@pytest.mark.gpu
@pytest.mark.parametrize("version", ["1.0", "2.0"])
def test_parquet_arrow_parquet_appends_of_one_boolean_column(ctx, tmp_path, version):
    """the host mirror of the value bitmap's last byte must follow the device appends: an Arrow append after a Parquet
    append at an unaligned row continues from it"""
    rng = np.random.default_rng(5)
    parts, pieces = [], []
    for k, n in enumerate((70_001, 3, 13, 5, 1, 9_999)):
        arr = pa.array(rng.random(n) < 0.5, mask=rng.random(n) < 0.2)
        pieces.append(arr)
        if k % 2 == 0:
            path = os.path.join(str(tmp_path), f"ap{k}.parquet")
            pq.write_table(pa.table({"b": arr}), path, data_page_version=version, compression="NONE", data_page_size=2048)
            parts.append(("pq", path))
        else:
            parts.append(("arrow", pa.record_batch([arr], names=["b"])))
    tab = ctx._create("mix")
    try:
        for kind, x in parts:
            if kind == "arrow":
                ctx._append_batch_c(tab, x)
                continue
            for _, name, chunk, cm, leaf in _chunks(x):
                F.check(F.lib().tg_table_append_parquet_chunk(tab, b"b", F.TG_BOOL, leaf.max_definition_level, 0, chunk.ctypes.data,
                                                              chunk.size, cm.num_values))
        _check_bool(ctx, "mix", "b", pa.concat_arrays(pieces), nulls_read_zero=False)
    finally:
        ctx.deregister_table("mix")


@pytest.mark.gpu
def test_int96_appended_to_another_type_is_refused(ctx, tmp_path):
    path, t = _write(tmp_path, 1000, 0.1, None, "1.0")
    (_, _, chunk, cm, leaf), = [c for c in _chunks(path) if c[1] == "ts"]
    for typ in (pa.int64(), pa.timestamp("us")):
        tab = ctx._create("i96")
        try:
            ctx._append_batch_c(tab, pa.record_batch([pa.array([1, 2, 3], type=typ)], names=["ts"]))
            st = F.lib().tg_table_append_parquet_chunk(tab, b"ts", F.TG_PQ_INT96, 1, 0, chunk.ctypes.data, chunk.size, cm.num_values)
            assert st == 3, (typ, st, F.last_error())  # TG_ERR_TYPE_MISMATCH
            assert ctx.num_rows("i96") == 3
        finally:
            ctx.deregister_table("i96")
    # INT96 after INT96, and after Arrow timestamp[ns], is one column
    tab = ctx._create("i96")
    try:
        ctx._append_batch_c(tab, pa.record_batch([pa.array([7], type=pa.timestamp("ns"))], names=["ts"]))
        for _ in range(2):
            F.check(F.lib().tg_table_append_parquet_chunk(tab, b"ts", F.TG_PQ_INT96, 1, 0, chunk.ctypes.data, chunk.size, cm.num_values))
        w = pq.read_table(path).column("ts").combine_chunks()
        _check_ts(ctx, "i96", "ts", pa.concat_arrays([pa.array([7], type=pa.timestamp("ns")), w, w]))
    finally:
        ctx.deregister_table("i96")


@pytest.mark.gpu
def test_suite_over_boolean_and_int96_parquet_equals_suite_over_arrow(ctx, tmp_path):
    path, _ = _write(tmp_path, 200_000, 0.05, 70_000, "2.0", "SNAPPY", 4096, seed=21)
    ctx.register_parquet("bi_pq", path)
    ctx.register_table("bi_ar", pq.read_table(path))
    try:
        A = T.Assertion

        def suite(name):
            cb = (T.Check.builder("c").completeness("b", 0.9).completeness("breq", 1.0).satisfies("b IS NOT TRUE").satisfies("NOT b AND x > 0")
                  .satisfies("b = true").satisfies("runs OR breq").validates_uniqueness(["b"], 0.0).validates_uniqueness(["b", "runs"], 0.0)
                  .validates_distinctness(["runs"], A.GreaterThan(0.0)).has_histogram("b", lambda h: h.bucket_count() <= 3)
                  .completeness("ts", 0.5).satisfies("ts >= TIMESTAMP '2001-01-01 00:00:00'").validates_uniqueness(["ts"], 0.0)
                  .validates_uniqueness(["tsc"], 0.0).has_min("ts", A.GreaterThan(0.0)).has_mean("ts", A.GreaterThan(0.0)))
            return [(r.name, r.status, r.metric, r.message) for r in
                    T.ValidationSuite.builder("s").table_name(name).check(cb.build()).build().run(ctx).report.results]
        got, want = suite("bi_pq"), suite("bi_ar")
        assert got == want, [(a, b) for a, b in zip(got, want) if a != b]
        maps = []
        for name in ("bi_pq", "bi_ar"):
            plan = T.Plan()
            slot = T.GroupedCompletenessAnalyzer("x", ["b"])._add_to(plan)
            plan.execute(ctx, name)
            maps.append(plan.analyzer_result(slot).map)
        assert maps[0] == maps[1] and len(maps[0]) >= 3
    finally:
        ctx.deregister_table("bi_pq")
        ctx.deregister_table("bi_ar")


@pytest.mark.gpu
def test_malformed_and_refused_boolean_chunks(ctx):
    """each returns its status, appends nothing, and leaves the table usable"""
    good_vals, good_bits = _rle_values([("rle", 10, 1), ("packed", [1, 0] * 8)])
    stream = good_vals[4:]
    cases = [  # (chunk, rows, status): 1 TG_ERR_INVALID_ARG, 5 TG_ERR_UNSUPPORTED
        (_page(b"\x05\x00", 26, 3), 26, 1),                                               # RLE length prefix cut short
        (_page((len(stream) + 40).to_bytes(4, "little") + stream, 26, 3), 26, 1),         # length prefix past the section
        (_page(good_vals, 40, 3), 40, 1),                                                 # runs end before the values do
        (_page((3).to_bytes(4, "little") + _varint((4 << 1) | 1) + b"\xff\xff", 32, 3), 32, 1),  # a bit-packed run past the stream
        (_page((2).to_bytes(4, "little") + _varint(26 << 1) + b"\x02", 26, 3), 26, 1),     # an RLE run of the value 2
        (_page(b"\xff", 26, 0), 26, 1),                                                   # PLAIN section shorter than 26 bits
        (_page(b"\xff" * 4, 26, 4), 26, 5),                                               # BIT_PACKED values
        (_page(b"\x01", 1, 0, page_type=2) + _page(b"\x00" + _varint(2 << 1), 2, 8), 2, 5),  # a dictionary-encoded BOOLEAN chunk
        (_page(b"\x00" * 16, 26, 5), 26, 5),                                              # DELTA_BINARY_PACKED values
    ]
    tab = ctx._create("bad")
    try:
        F.check(_append_chunk(tab, "b", F.TG_BOOL, 0, _page(good_vals, 26, 3), 26))
        for chunk, n, want in cases:
            st = _append_chunk(tab, "b", F.TG_BOOL, 0, chunk, n)
            assert st == want, (chunk[:24], st, F.last_error())
            assert ctx.num_rows("bad") == 26
        F.check(_append_chunk(tab, "b", F.TG_BOOL, 0, _page(good_vals, 26, 3), 26))
        _check_bool(ctx, "bad", "b", pa.array(np.concatenate([good_bits, good_bits])))
    finally:
        ctx.deregister_table("bad")


@pytest.mark.gpu
def test_full_size_boolean_column_counts(ctx, tmp_path):
    n = 100_000_000
    rng = np.random.default_rng(100)
    t = pa.table({"b": pa.array(rng.random(n) < 0.37, mask=rng.random(n) < 0.02)})
    path = os.path.join(str(tmp_path), "big_bool.parquet")
    pq.write_table(t, path, compression="SNAPPY", data_page_version="2.0")
    ctx.register_parquet("bigb", path)
    try:
        vals, valid, b = _read(ctx, "bigb", "b")
        bits = np.unpackbits(vals, bitorder="little")[:n].astype(bool)
        col = t.column("b")
        assert int((bits & valid).sum()) == pc.sum(col).as_py()
        assert int((~bits & valid).sum()) == pc.sum(pc.invert(col)).as_py()
        assert int((~valid).sum()) == col.null_count == b["null_count"]
        assert not bits[~valid].any()
    finally:
        ctx.deregister_table("bigb")
