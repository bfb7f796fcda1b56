"""CSV ingestion: tg_table_append_csv tokenizes and parses whole records on the GPU into the Arrow layout. CPU tests pin the
value parser the device runs (tg_csv_parse_value) against Python — Float64 bit for bit against float() — and the generated
power-of-five table. GPU tests compare the decoded buffers with pyarrow's CSV reader (which agrees with the format contract
on the files written here), cut the same files into chunks of a few KiB, append CSV and Arrow to one column, run a suite
over both registrations, check every error class and that a failed append changes nothing, and read a ~1 GB file."""
import ctypes as C
import datetime as dt
import os
import random
import struct
import subprocess
import sys

import numpy as np
import pyarrow as pa
import pyarrow.csv as pacsv
import pytest

import term_b200 as T
from term_b200 import _ffi as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pv(fmt, field):
    """(status, value, is_null) of tg_csv_parse_value"""
    b = field.encode() if isinstance(field, str) else field
    out = (C.c_uint8 * 8)()
    isn = C.c_int32()
    st = F.lib().tg_csv_parse_value(fmt.encode(), b, len(b), out, C.byref(isn))
    raw = bytes(out)
    if fmt in ("i", "tdD"):
        v = struct.unpack("<i", raw[:4])[0]
    elif fmt == "b":
        v = raw[0]
    elif fmt == "g":
        v = struct.unpack("<Q", raw)[0]
    else:
        v = struct.unpack("<q", raw)[0]
    return st, v, bool(isn.value)


def _bits(x):
    return struct.unpack("<Q", struct.pack("<d", x))[0]


# ------------------------------------------------------------------------------------------ CPU ----
def test_float64_parse_is_correctly_rounded(built_lib):
    rng = random.Random(20261020)
    fixed = ["9007199254740993", "9007199254740992.5", "1e400", "-1e400", "1e-400", "-1e-400", "-0.0", "0", "0.0e-999", "1e-999999999",
             "2.2250738585072011e-308", "2.2250738585072014e-308", "2.2250738585072009e-308", "4.9406564584124654e-324",
             "2.4703282292062327e-324", "2.4703282292062328e-324", "2.4703282292062328e-324", "1.7976931348623157e308",
             "1.7976931348623158e308", "1.7976931348623159e308", "179769313486231580793728971405301e276", ".5", "5.", "+1e+3", "-.25E-2",
             "1.00000000000000011102230246251565404236316680908203125", "1.00000000000000011102230246251565404236316680908203124",
             "0." + "0" * 400 + "1e400", "1" + "0" * 400 + "e-400", "123456789012345678901234567890"]
    strs = list(fixed)
    while len(strs) < 1_000_000:
        x = struct.unpack("<d", struct.pack("<Q", rng.getrandbits(64)))[0]
        if x != x or x in (float("inf"), float("-inf")):
            continue
        sub = struct.unpack("<d", struct.pack("<Q", rng.getrandbits(52)))[0]  # subnormals
        strs += [repr(x), "%.17g" % x, "%.25e" % x, "%.3f" % rng.uniform(-1e6, 1e6), repr(sub), "%.25e" % sub,
                 f"{rng.getrandbits(53) * 2 + 1}e{rng.randint(-330, 290)}"]
    bad = []
    for s in strs:
        st, v, isn = _pv("g", s)
        if st != 0 or isn or v != _bits(float(s)):
            bad.append((s, st, v, _bits(float(s))))
    assert not bad, (len(bad), bad[:5])
    assert _pv("g", "nan")[1] == 0x7FF8000000000000 and _pv("g", "-NaN")[1] == 0xFFF8000000000000
    assert _pv("g", "Infinity")[1] == _bits(float("inf")) and _pv("g", "-inf")[1] == _bits(float("-inf"))
    for s in ["1e", "e5", ".", "1.2.3", " 1", "1 ", "0x10", "1_0", "--1", "+", "nanx", "in", "1e+", "1.5f"]:
        assert _pv("g", s)[0] == 1, s  # TG_ERR_INVALID_ARG
    assert F.lib().tg_csv_parse_value(b"g", b"x1", 2, None, None) == 1 and "cannot parse 'x1' as Float64" in F.last_error()


def test_integer_boolean_date_and_quoting(built_lib):
    for fmt, lo, hi in (("l", -2**63, 2**63 - 1), ("i", -2**31, 2**31 - 1)):
        for v in (lo, hi, 0, -1, 1):
            assert _pv(fmt, str(v))[:2] == (0, v)
        for s in (str(lo - 1), str(hi + 1), "99999999999999999999999"):
            st, _, _ = _pv(fmt, s)
            assert st == 1 and "out of range" in F.last_error(), s
        for s in ("", '""'):
            assert _pv(fmt, s)[2], s
        for s in ("1a", "-", "1.0", " 1", "0x1", '"1""2"'):
            assert _pv(fmt, s)[0] == 1, s
    assert _pv("l", "+5")[1] == 5 and _pv("l", '"42"')[1] == 42 and _pv("l", '"4"2')[1] == 42
    for s, v in (("true", 1), ("TRUE", 1), ("tRuE", 1), ("false", 0), ("False", 0), ("FALSE", 0)):
        assert _pv("b", s)[:2] == (0, v)
    for s in ("yes", "1", "t", "truee", " true"):
        assert _pv("b", s)[0] == 1
    epoch = dt.date(1970, 1, 1)
    for d in ("2020-02-29", "2000-02-29", "1969-12-31", "0001-01-01", "9999-12-31", "1900-03-01"):
        assert _pv("tdD", d)[:2] == (0, (dt.date.fromisoformat(d) - epoch).days), d
    for d in ("2019-02-29", "1900-02-29", "2021-04-31", "2020-13-01", "2020-1-01", "2020-01-01T00:00:00", "20200101"):
        assert _pv("tdD", d)[0] == 1, d


@pytest.mark.parametrize("unit,per_s", [("s", 1), ("m", 1000), ("u", 10**6), ("n", 10**9)])
def test_timestamps_before_and_after_1970_with_every_fraction_length(built_lib, unit, per_s):
    rng = random.Random(7)
    base = dt.datetime(1970, 1, 1)
    for _ in range(300):
        secs = rng.randint(-2_000_000_000, 2_000_000_000)
        t = base + dt.timedelta(seconds=secs)
        digits = "".join(rng.choice("0123456789") for _ in range(9))
        for k in range(0, 10):
            s = t.strftime("%Y-%m-%d") + rng.choice("T ") + t.strftime("%H:%M:%S") + ("." + digits[:k] if k else "")
            frac = int((digits[:k] + "0" * 9)[:9])  # nanoseconds
            want = secs * per_s + frac * per_s // 10**9  # fraction digits past the unit dropped: floor
            assert _pv(f"ts{unit}:", s)[:2] == (0, want), s
    for s in ("2020-01-01 00:00:00Z", "2020-01-01 00:00:00+01:00", "2020-01-01 00:00:00.", "2020-01-01 24:00:00", "2020-01-01 00:60:00",
              "2020-01-01", "2020-01-01 00:00:00.1234567890"):
        assert _pv(f"ts{unit}:", s)[0] == 1, s


def test_utf8_validation_and_unescaping(built_lib):
    good = [b"abc", "é".encode(), "€".encode(), "😀".encode(), b"\xf4\x8f\xbf\xbf", b"\xef\xbf\xbd", b'"a""b"', b'"a,b\nc"', b'"ab"cd', b'ab"c']
    lens = [3, 2, 3, 4, 4, 3, 3, 5, 4, 4]
    for g, n in zip(good, lens):
        out = C.c_int64()
        assert F.lib().tg_csv_parse_value(b"u", g, len(g), C.byref(out), None) == 0, g
        assert out.value == n, g
    # Markus Kuhn's malformed sequences: overlong forms, surrogates, > U+10FFFF, lone / missing continuation bytes, 0xFE / 0xFF
    bad = [b"\xc0\xaf", b"\xe0\x80\xaf", b"\xf0\x80\x80\xaf", b"\xc1\xbf", b"\xe0\x9f\xbf", b"\xed\xa0\x80", b"\xed\xbf\xbf",
           b"\xf4\x90\x80\x80", b"\xf5\x80\x80\x80", b"\x80", b"\xbf", b"\xc3", b"\xe2\x82", b"\xf0\x9f\x98", b"\xfe", b"\xff", b"a\xc3(b"]
    for b in bad:
        assert F.lib().tg_csv_parse_value(b"u", b, len(b), None, None) == 1 and "invalid UTF-8" in F.last_error(), b
    assert _pv("u", '""')[2] and _pv("u", "")[2] and not _pv("u", '""""')[2]


def test_unsupported_formats_name_the_type(built_lib):
    for fmt, name in (("f", "Float32"), ("d:10,2", "Decimal"), ("tsu:UTC", "Timestamp(Microsecond, Some(\"UTC\"))"), ("C", "UInt8"),
                      ("s", "Int16"), ("L", "UInt64"), ("tdm", "Date64")):
        assert F.lib().tg_csv_parse_value(fmt.encode(), b"1", 1, None, None) == F.TG_ERR_UNSUPPORTED
        assert name in F.last_error(), (fmt, F.last_error())


def test_pow5_table_is_generated_and_exact(tmp_path):
    out = tmp_path / "pow5.inc"
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_pow5_table.py"), str(out)], check=True)
    committed = open(os.path.join(ROOT, "term_b200", "csrc", "pow5_128.inc"), "rb").read()
    assert out.read_bytes() == committed
    rows = [ln.strip() for ln in committed.decode().splitlines() if ln.strip().startswith("{")]
    assert len(rows) == 308 + 342 + 1
    for i, ln in enumerate(rows):
        q = i - 342
        hi, lo = (int(x.strip().rstrip("ull"), 16) for x in ln.strip("{},").split(","))
        v = (hi << 64) | lo
        if q >= 0:  # the top 128 bits of 5^q
            p = 5 ** q
            want = p << (128 - p.bit_length()) if p.bit_length() <= 128 else p >> (p.bit_length() - 128)
        else:  # the top 128 bits of 1 / 5^-q, rounded up
            p = 5 ** -q
            z = (p - 1).bit_length()
            c = (1 << (z + 127 if q >= -27 else 2 * z + 128)) // p + 1
            want = c >> max(0, c.bit_length() - 128)
        assert v == want and v >> 127 == 1, q


# ------------------------------------------------------------------------------------------ GPU ----
SCHEMA = pa.schema([pa.field("i64", pa.int64()), pa.field("i32", pa.int32()), pa.field("f64", pa.float64()), pa.field("flag", pa.bool_()),
                    pa.field("s", pa.string()), pa.field("d", pa.date32()), pa.field("ts", pa.timestamp("us")), pa.field("tss", pa.timestamp("s"))])
WORDS = ["alpha", "b,c", 'say "hi"', "line\nbreak", "crlf\r\nin", "ünï", "日本", "semi;colon", "tab\tx", "pipe|y", "x@example.com", "plain"]


def _rows(n, null_p, seed):
    rng = np.random.default_rng(seed)
    base = dt.datetime(1970, 1, 1)
    rows = []
    for i in range(n):
        def nul():
            return rng.random() < null_p
        secs = int(rng.integers(-1_500_000_000, 2_000_000_000))
        us = int(rng.integers(0, 10**6))
        t = base + dt.timedelta(seconds=secs, microseconds=us)
        rows.append([
            None if nul() else int(rng.integers(-2**62, 2**62)),
            None if nul() else int(rng.integers(-2**31, 2**31)),
            None if nul() else float(rng.normal(0, 1e3)) if i % 7 else float(rng.choice([0.1, -0.0, 1e300, 5e-324, 123.0])),
            None if nul() else bool(rng.random() < 0.5),
            None if nul() else WORDS[int(rng.integers(0, len(WORDS)))] + str(i),
            None if nul() else (base + dt.timedelta(days=int(rng.integers(-30000, 30000)))).date(),
            None if nul() else t,
            None if nul() else base + dt.timedelta(seconds=secs),
        ])
    return rows


def _field(v, delim, k):
    if v is None:
        return "" if k % 2 else '""'  # empty, quoted or not: NULL
    if isinstance(v, bool):
        s = ("true", "FALSE", "True", "false")[k % 4] if v else ("false", "False", "FALSE")[k % 3]
    elif isinstance(v, float):
        s = repr(v)
    elif isinstance(v, dt.datetime):
        s = v.isoformat(sep="T" if k % 2 else " ")
    elif isinstance(v, dt.date):
        s = v.isoformat()
    else:
        s = str(v)
    if any(c in s for c in (delim, '"', "\n", "\r")) or k % 5 == 0:
        return '"' + s.replace('"', '""') + '"'
    return s


def _write_csv(path, rows, delim=",", eol="\n", header=True, final_eol=True, blank_lines=False):
    lines = []
    if header:
        lines.append(delim.join(f.name for f in SCHEMA))
    for i, r in enumerate(rows):
        lines.append(delim.join(_field(v, delim, i + j) for j, v in enumerate(r)))
        if blank_lines and i % 97 == 5:
            lines.append("")
    text = eol.join(lines) + (eol if final_eol else "")
    with open(path, "w", newline="", encoding="utf-8") as f:
        f.write(text)


def _pyarrow_read(path, schema, delim=",", header=True):
    ro = pacsv.ReadOptions(column_names=[f.name for f in schema], skip_rows=1 if header else 0, block_size=1 << 20)
    po = pacsv.ParseOptions(delimiter=delim, newlines_in_values=True)
    co = pacsv.ConvertOptions(column_types=schema, strings_can_be_null=True, quoted_strings_can_be_null=True, null_values=[""],
                              true_values=["true", "True", "TRUE"], false_values=["false", "False", "FALSE"])
    return pacsv.read_csv(path, read_options=ro, parse_options=po, convert_options=co)


def _read(ctx, table, column):
    """(buffers dict, validity bool ndarray, values bytes, offsets) of a device column"""
    import torch
    from term_b200.distributed import _tensor_from_ptr
    b = ctx.column_buffers(table, column)
    dev = torch.device("cuda", 0)
    n = b["n_rows"]
    get = lambda p, k: _tensor_from_ptr(p, max(k, 1), dev, "|u1").cpu().numpy()[:k]  # noqa: E731
    if b["validity"]:
        valid = np.unpackbits(get(b["validity"], (n + 7) // 8), bitorder="little")[:n].astype(bool)
    else:
        valid = np.ones(n, dtype=bool)
    offs = None
    if b["dtype"] == F.TG_UTF8:
        offs = get(b["offsets"], 4 * (n + 1)).view(np.int32)
        vals = get(b["values"], b["n_value_bytes"])
    elif b["dtype"] == F.TG_BOOL:
        vals = get(b["values"], (n + 7) // 8)
    else:
        vals = get(b["values"], n * (8 if b["dtype"] in (F.TG_INT64, F.TG_FLOAT64) else 4))
    return b, valid, vals, offs


def _check_table(ctx, name, want):
    """every column's buffers against pyarrow's read: validity, NULL count, values of valid rows, Utf8 offsets and bytes"""
    for col in want.column_names:
        a = want.column(col).combine_chunks()
        b, valid, vals, offs = _read(ctx, name, col)
        n = len(a)
        assert b["n_rows"] == n, col
        wv = np.asarray(a.is_valid())
        assert (valid == wv).all(), col
        assert b["null_count"] == a.null_count, col
        if pa.types.is_string(a.type):
            wo = np.frombuffer(a.buffers()[1], dtype=np.int32)[a.offset: a.offset + n + 1]
            o0 = int(wo[0])
            wo = wo - o0
            assert (offs == wo).all(), col
            assert vals.tobytes() == bytes(a.buffers()[2])[o0: o0 + int(wo[-1])], col
        elif pa.types.is_boolean(a.type):
            got = np.unpackbits(vals, bitorder="little")[:n].astype(bool)
            wb = np.asarray(a.fill_null(False))
            assert (got[wv] == wb[wv]).all(), col
        else:
            w = 8 if a.type.bit_width == 64 else 4
            g = vals.view(np.int64 if w == 8 else np.int32)
            wa = np.frombuffer(a.buffers()[1], dtype=np.int64 if w == 8 else np.int32)[a.offset: a.offset + n]
            assert (g[wv] == wa[wv]).all(), col


def _register(ctx, name, path, schema=SCHEMA, **kw):
    ctx.register_csv(name, path, schema, **kw)
    return name


@pytest.mark.gpu
@pytest.mark.parametrize("null_p", [0.0, 0.05, 1.0])
@pytest.mark.parametrize("delim,eol,header,final_eol,blank", [(",", "\n", True, True, False), (";", "\r\n", False, False, True),
                                                               ("\t", "\r", True, False, False), ("|", "\n", False, True, True)])
def test_decoded_buffers_equal_pyarrow(ctx, tmp_path, null_p, delim, eol, header, final_eol, blank):
    path = str(tmp_path / "t.csv")
    _write_csv(path, _rows(3000, null_p, 3), delim, eol, header, final_eol, blank)
    want = _pyarrow_read(path, SCHEMA, delim, header)
    _register(ctx, "csv_t", path, delimiter=delim, has_header=header)
    try:
        assert ctx.num_rows("csv_t") == 3000
        _check_table(ctx, "csv_t", want)
    finally:
        ctx.deregister_table("csv_t")


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [1024, 4093, 8192, 65537])
def test_small_chunks_give_the_same_columns(ctx, tmp_path, monkeypatch, chunk):
    # records and quoted line breaks straddle the chunk edges; one record is longer than a chunk
    rows = _rows(2000, 0.05, 5)
    rows[777][4] = "long " + "x,\"y\"\n" * 3000
    path = str(tmp_path / "c.csv")
    _write_csv(path, rows, ",", "\r\n", True, False, True)
    want = _pyarrow_read(path, SCHEMA)
    monkeypatch.setenv("TG_CSV_CHUNK_BYTES", str(chunk))  # read at every call
    ctx.register_csv("small", path, SCHEMA)
    try:
        assert ctx.num_rows("small") == want.num_rows == 2000
        _check_table(ctx, "small", want)
    finally:
        ctx.deregister_table("small")


@pytest.mark.gpu
def test_csv_and_arrow_appends_at_unaligned_rows(ctx, tmp_path):
    schema = pa.schema([pa.field("x", pa.float64()), pa.field("flag", pa.bool_())])
    rng = np.random.default_rng(11)
    parts = []
    tab = ctx._create("mix")
    try:
        for k, n in enumerate([13, 1001, 7, 333, 64, 5]):
            x = pa.array(rng.normal(0, 1, n), mask=rng.random(n) < 0.3)
            fl = pa.array(rng.random(n) < 0.5, mask=rng.random(n) < (0.0 if k == 0 else 0.2))
            t = pa.table({"x": x, "flag": fl})
            parts.append(t)
            if k % 2 == 0:
                p = str(tmp_path / f"m{k}.csv")
                pacsv.write_csv(t, p, pacsv.WriteOptions(include_header=False))
                with open(p, "rb") as f:
                    data = f.read()
                names, _ = T.api._strs(["x", "flag"])
                fmts, _ = T.api._strs(["g", "b"])
                rows = C.c_int64()
                F.check(F.lib().tg_table_append_csv(tab, names, fmts, 2, data, len(data), ord(","), 0, C.byref(rows)))
                assert rows.value == n
            else:
                ctx._append_batch(tab, t.to_batches()[0], False)
        _check_table(ctx, "mix", pa.concat_tables(parts))
    finally:
        ctx.deregister_table("mix")


def _suite(ctx, name):
    A = T.Assertion
    cb = (T.Check.builder("c").completeness("i64", 0.9).completeness("s", 0.5).has_min("f64", A.LessThan(0.0)).has_max("i64", A.GreaterThan(0.0))
          .has_mean("f64", A.Between(-100.0, 100.0)).has_sum("i32", A.GreaterThan(-1e30)).has_standard_deviation("f64", A.GreaterThan(0.0))
          .validates_uniqueness(["i64"], 0.5).validates_uniqueness(["flag", "d"], 0.0).validates_email("s", 0.01)
          .validates_regex("s", "^[a-z]+[0-9]+$", 0.1).satisfies("flag OR i32 > 0").completeness("ts", 0.9)
          .constraint(T.TemporalOrderingConstraint(name).before_after("tss", "ts"))
          .constraint(T.QuantileConstraint.median("f64", A.Between(-1e6, 1e6))))
    res = T.ValidationSuite.builder("s").table_name(name).check(cb.build()).build().run(ctx).report.results
    plan = T.Plan()
    slot = T.GroupedCompletenessAnalyzer("i32", ["flag"])._add_to(plan)
    plan.execute(ctx, name)
    return [(r.name, r.status, r.metric, r.message) for r in res], plan.analyzer_result(slot).map


@pytest.mark.gpu
def test_suite_over_csv_equals_suite_over_arrow(ctx, tmp_path):
    path = str(tmp_path / "s.csv")
    _write_csv(path, _rows(20000, 0.05, 9))
    ctx.register_csv("s_csv", path, SCHEMA)
    ctx.register_table("s_arrow", _pyarrow_read(path, SCHEMA))
    try:
        got, want = _suite(ctx, "s_csv"), _suite(ctx, "s_arrow")
        assert got[0] == want[0], [(a, b) for a, b in zip(got[0], want[0]) if a != b]
        assert got[1] == want[1] and len(got[1]) >= 2
    finally:
        ctx.deregister_table("s_csv")
        ctx.deregister_table("s_arrow")


ERRORS = [  # (file text, schema of (name, format), status, message part)
    ("a,b\n1,2\n3\n", [("a", "l"), ("b", "l")], 1, "CSV line 3, column 'b': missing"),
    ("a,b\n1,2\n3,4,5\n", [("a", "l"), ("b", "l")], 1, "CSV line 3, column 'b': followed by an extra field"),
    ('a,b\n1,"x\ny"\n2,"open\n\nend', [("a", "l"), ("b", "u")], 1, "CSV line 4, column 'b': unterminated quote"),
    ('a,b\n1,"two\nlines"\n2,3\nx1,4\n', [("a", "g"), ("b", "u")], 1, "CSV line 5, column 'a': cannot parse 'x1' as Float64"),
    ("a\n1\r\n\r\n99999999999\n", [("a", "i")], 1, "CSV line 4, column 'a': '99999999999' is out of range for Int32"),
    (b"a,b\n1,ok\n2,\xc0\xaf\n", [("a", "l"), ("b", "u")], 1, "CSV line 3, column 'b': invalid UTF-8"),
    ("a\n2020-02-30\n", [("a", "tdD")], 1, "CSV line 2, column 'a': cannot parse '2020-02-30' as Date32"),
    ("a\n2020-01-01T00:00:00Z\n", [("a", "tsu:")], 1, "Timestamp(Microsecond, None)"),
    ("a\n1\n", [("a", "f")], F.TG_ERR_UNSUPPORTED, "Float32"),
    ("a\n1\n", [("a", "tsu:UTC")], F.TG_ERR_UNSUPPORTED, "Timestamp(Microsecond, Some(\"UTC\"))"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [None, 5, 8, 13])  # (chunks of a few bytes: every record straddles a chunk edge somewhere)
@pytest.mark.parametrize("k", range(len(ERRORS)))
def test_errors_name_line_and_column_and_change_nothing(ctx, monkeypatch, k, chunk):
    if chunk:
        monkeypatch.setenv("TG_CSV_CHUNK_BYTES", str(chunk))
    text, cols, status, msg = ERRORS[k]
    data = text.encode() if isinstance(text, str) else text
    schema = [(n, f) for n, f in cols]
    tab = ctx._create("err")
    try:
        # the table already holds rows of every column (CSV with the same schema); a failed append leaves it unchanged
        good = ",".join(n for n, _ in schema) + "\n" + ",".join({"l": "5", "i": "6", "g": "1.5", "u": "ok", "tdD": "2001-02-03",
                                                                    "tsu:": "2001-02-03 04:05:06"}.get(f, "") for _, f in schema) + "\n"
        names, _ = T.api._strs([n for n, _ in schema])
        fmts, _ = T.api._strs([f for _, f in schema])
        rows = C.c_int64()
        supported = status != F.TG_ERR_UNSUPPORTED
        if supported:
            gb = good.encode()
            F.check(F.lib().tg_table_append_csv(tab, names, fmts, len(schema), gb, len(gb), ord(","), 1, C.byref(rows)))
        before = [_read(ctx, "err", n)[1:] for n, _ in schema] if supported else []
        st = F.lib().tg_table_append_csv(tab, names, fmts, len(schema), data, len(data), ord(","), 1, C.byref(rows))
        assert st == status, (st, F.last_error())
        assert msg in F.last_error(), F.last_error()
        if supported:
            assert ctx.num_rows("err") == 1
            after = [_read(ctx, "err", n)[1:] for n, _ in schema]
            for (v0, b0, o0), (v1, b1, o1) in zip(before, after):
                assert (v0 == v1).all() and b0.tobytes() == b1.tobytes() and (o0 is None or (o0 == o1).all())
            # and the table still appends
            F.check(F.lib().tg_table_append_csv(tab, names, fmts, len(schema), gb, len(gb), ord(","), 1, C.byref(rows)))
            assert ctx.num_rows("err") == 2
    finally:
        ctx.deregister_table("err")


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [None, 3, 4, 5, 6, 7, 8, 9, 10, 11])
def test_short_record_at_a_chunk_edge_is_an_error(ctx, monkeypatch, chunk):
    # a record with too few fields that ends a chunk's last complete line must not be skipped by the next chunk
    if chunk:
        monkeypatch.setenv("TG_CSV_CHUNK_BYTES", str(chunk))
    tab = ctx._create("edge")
    try:
        names, _ = T.api._strs(["a", "b"])
        fmts, _ = T.api._strs(["l", "l"])
        for data, line in ((b"1,2\n3\n4,5\n", 2), (b"1,2\n3,4\n5\n6,7\n8,9\n", 3), (b"1,2\r\n\r\n3\r\n4,5", 3)):
            st = F.lib().tg_table_append_csv(tab, names, fmts, 2, data, len(data), ord(","), 0, None)
            assert st == 1 and f"CSV line {line}, column 'b': missing" in F.last_error(), (data, F.last_error())
            assert ctx.num_rows("edge") == 0
    finally:
        ctx.deregister_table("edge")


@pytest.mark.gpu
def test_temporal_append_needs_the_same_delivered_type(ctx):
    tab = ctx._create("tt")
    try:
        ctx._append_batch_c(tab, pa.record_batch([pa.array([7], type=pa.date64()), pa.array([1], type=pa.timestamp("us"))], names=["d", "t"]))
        for col, fmt in (("d", "tsm:"), ("t", "tsm:"), ("t", "l"), ("d", "l")):
            names, _ = T.api._strs([col])
            fmts, _ = T.api._strs([fmt])
            data = b"1\n" if fmt == "l" else b"2001-01-01 00:00:00\n"
            assert F.lib().tg_table_append_csv(tab, names, fmts, 1, data, len(data), ord(","), 0, None) == 3, (col, fmt, F.last_error())
        names, _ = T.api._strs(["t"])
        fmts, _ = T.api._strs(["tsu:"])
        data = b"2001-01-01 00:00:00.000001\n"
        F.check(F.lib().tg_table_append_csv(tab, names, fmts, 1, data, len(data), ord(","), 0, None))
        assert ctx.column_buffers("tt", "t")["n_rows"] == 2
    finally:
        ctx.deregister_table("tt")


@pytest.mark.gpu
def test_failed_append_leaves_suite_results_unchanged(ctx, tmp_path):
    path = str(tmp_path / "ok.csv")
    _write_csv(path, _rows(5000, 0.05, 13))
    ctx.register_csv("fa", path, SCHEMA)
    try:
        before = _suite(ctx, "fa")
        bad = str(tmp_path / "bad.csv")
        rows = _rows(3000, 0.2, 14)
        _write_csv(bad, rows)
        with open(bad, "a") as f:
            f.write("1,2,notafloat,true,x,2001-01-01,2001-01-01 00:00:00,2001-01-01 00:00:00\n")
        with open(bad, "rb") as f:
            data = f.read()
        t = C.c_void_p()
        F.check(F.lib().tg_table_lookup(ctx.handle, b"fa", C.byref(t)))
        names, _ = T.api._strs([f.name for f in SCHEMA])
        fmts, _ = T.api._strs([T.api._arrow_format(f.type) for f in SCHEMA])
        st = F.lib().tg_table_append_csv(t, names, fmts, len(SCHEMA), data, len(data), ord(","), 1, None)
        assert st == 1 and "column 'f64': cannot parse 'notafloat' as Float64" in F.last_error(), F.last_error()
        assert _suite(ctx, "fa") == before
    finally:
        ctx.deregister_table("fa")


@pytest.mark.gpu
def test_full_size_file_spans_several_chunks(ctx, tmp_path):
    # ~1 GB: Int64, Float64 and C3-shaped Utf8 (emails, some quoted with a comma) over 20 M rows, several 256 MiB chunks
    n = 20_000_000
    rng = np.random.default_rng(42)
    ids = rng.integers(-10**15, 10**15, n)
    xs = rng.normal(100.0, 15.0, n)
    path = str(tmp_path / "big.csv")
    schema = pa.schema([pa.field("id", pa.int64()), pa.field("x", pa.float64()), pa.field("email", pa.string())])
    step = 1_000_000
    with open(path, "w") as f:
        f.write("id,x,email\n")
        for lo in range(0, n, step):
            idx = np.arange(lo, min(n, lo + step))
            em = np.where(idx % 10 == 0, np.char.add(np.char.add('"user', idx.astype(str)), ',x@example.com"'),
                          np.char.add(np.char.add("user", idx.astype(str)), "@example.com"))
            em = np.where(idx % 101 == 0, "", em)
            lines = np.char.add(np.char.add(np.char.add(np.char.add(ids[idx].astype(str), ","), np.char.mod("%.17g", xs[idx])), ","), em)
            f.write("\n".join(lines.tolist()) + "\n")
    assert os.path.getsize(path) > 700 << 20
    ctx.register_csv("big", path, schema)
    try:
        _check_table(ctx, "big", _pyarrow_read(path, schema))
    finally:
        ctx.deregister_table("big")
