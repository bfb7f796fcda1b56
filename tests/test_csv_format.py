"""CSV dialects: quote, escape, comment and terminator bytes and a NULL regex (tg_table_append_csv_format, register_csv's
options). A Python restatement of csv-core's reader is the reference. On the CPU it is cross-checked against pyarrow's
reader where the two agree, and tg_csv_split_host (the tokenizer's transition table and the field rules run on the host)
must equal it on fuzzed inputs. On the GPU every stored type is decoded against the reference's parse across a matrix of
dialects, at the default chunk size and at chunks of a few KiB and a few bytes; the default dialect gives the same
buffers as tg_table_append_csv; errors name their line and change nothing; a suite over a dump-style file equals the suite
over the same data registered from Arrow; and a ~1 GB dump-style file is read."""
import ctypes as C
import io
import os
import random
import re

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc
import pyarrow.csv as pacsv
import pytest

import term_b200 as T
from term_b200 import _ffi as F
from tests.test_csv import SCHEMA, _check_table, _read, _rows, _suite

INVALID_ARG = 1  # TG_ERR_INVALID_ARG


# ------------------------------------------------------------------------------------ reference ----
def model(data, delimiter=",", quote='"', escape=None, comment=None, terminator=None, null=None):
    """csv-core's reader: [(line of the record's first byte, [(value bytes, is NULL)])], the state before every byte, and
    the error ("unterminated", line) or None. `null` is a function of the unescaped value (None: the value is empty)."""
    D, Q = ord(delimiter), ord(quote)
    E = ord(escape) if escape else -1
    M = ord(comment) if comment else -1
    if terminator:
        Tb = ord(terminator)
        is_term = lambda b: b == Tb  # noqa: E731
    else:
        is_term = lambda b: b in (10, 13)  # noqa: E731
    ends = [(b == Tb) if terminator else (b == 10 or (b == 13 and not (i + 1 < len(data) and data[i + 1] == 10)))
            for i, b in enumerate(data)]
    lines = np.concatenate([[1], 1 + np.cumsum(np.array(ends, dtype=np.int64))]) if data else np.array([1])
    recs, fields, field, states = [], [], bytearray(), []
    st, rec_line = "rec", 1

    def end_field():
        nonlocal field
        v = bytes(field)
        fields.append((v, null(v) if null else v == b""))
        field = bytearray()

    def end_record():
        nonlocal fields
        end_field()
        recs.append((rec_line, fields))
        fields = []

    for i, b in enumerate(data):
        states.append(st)
        if st == "rec":
            if is_term(b):
                continue
            if b == M:
                st = "cmt"
                continue
            rec_line = int(lines[i])
            st = "field"
        if st == "cmt":
            if is_term(b):
                st = "rec"
        elif st == "field":
            if b == Q:
                st = "quo"
            elif b == D:
                end_field()
            elif is_term(b):
                end_record()
                st = "rec"
            else:
                field.append(b)
                st = "unq"
        elif st == "unq":
            if b == D:
                end_field()
                st = "field"
            elif is_term(b):
                end_record()
                st = "rec"
            else:
                field.append(b)
        elif st == "quo":
            if b == Q:
                st = "qseen"
            elif b == E:
                st = "esc"
            else:
                field.append(b)
        elif st == "esc":
            field.append(b)
            st = "quo"
        else:  # qseen
            if b == Q:
                field.append(b)
                st = "quo"
            elif b == D:
                end_field()
                st = "field"
            elif is_term(b):
                end_record()
                st = "rec"
            else:
                field.append(b)
                st = "unq"
    if st in ("quo", "esc"):
        return recs, states, ("unterminated", rec_line)
    if st in ("field", "unq", "qseen"):
        end_record()
    return recs, states, None


NULL_RX = {None: None, "dump": r"^(NA|\\N|null)$", "empty": r"^(NA)?$"}
NULL_PY = {None: None, "dump": lambda v: re.search(rb"^(NA|\\N|null)\Z", v) is not None, "empty": lambda v: re.search(rb"^(NA)?\Z", v) is not None}


def fmt_of(delimiter=",", quote='"', escape=None, comment=None, terminator=None, null_regex=None, has_header=True):
    return T.api.csv_format(delimiter, quote, escape, comment, terminator, null_regex, has_header)


def split_host(data, **kw):
    """tg_csv_split_host: (status, records as the model gives them, or the error message)"""
    n = len(data)
    vals = (C.c_uint8 * max(n, 1))()
    ends, isn = (C.c_int64 * (n + 1))(), (C.c_uint8 * (n + 1))()
    rf, rl = (C.c_int64 * (n + 1))(), (C.c_int64 * (n + 1))()
    nf, nr = C.c_int64(), C.c_int64()
    f = fmt_of(**kw)
    st = F.lib().tg_csv_split_host(C.byref(f), data, n, vals, ends, isn, rf, rl, C.byref(nf), C.byref(nr))
    if st:
        return st, F.last_error()
    raw = bytes(vals)
    recs, k, o = [], 0, 0
    for r in range(nr.value):
        fs = []
        for _ in range(rf[r]):
            fs.append((raw[o:ends[k]], bool(isn[k])))
            o = ends[k]
            k += 1
        recs.append((rl[r], fs))
    return 0, recs


# ------------------------------------------------------------------------------------------ CPU ----
def test_model_agrees_with_pyarrow_where_both_readers_agree():
    # escape bytes only inside quotes, no comments, default terminators: csv-core's rules and pyarrow's coincide
    rng = random.Random(5)
    for trial in range(300):
        quote = rng.choice(['"', "'"])
        escape = rng.choice([None, "\\"])
        K = rng.randint(1, 4)
        eol = rng.choice(["\n", "\r\n", "\r"])
        lines = []
        for _ in range(rng.randint(1, 12)):
            fs = []
            for _ in range(K):
                s = "".join(rng.choice(["a", "b", ",", quote, "\\", "\n", "\r", "N", "x y"]) for _ in range(rng.randint(0, 6)))
                if rng.random() < 0.15:
                    s = rng.choice(["NA", "null", "\\N"])
                if not s or rng.random() < 0.5 or any(c in s for c in (",", quote, "\\", "\n", "\r")):
                    body = "".join((escape + c if escape and rng.random() < 0.5 else c + c) if c == quote else
                                   (escape + c if escape and (c == escape or rng.random() < 0.2) else c) for c in s)
                    s = quote + body + quote
                fs.append(s)
            lines.append(",".join(fs))
        data = (eol.join(lines) + (eol if rng.random() < 0.5 else "")).encode()
        recs, _, err = model(data, quote=quote, escape=escape, null=NULL_PY["dump"])
        assert err is None
        if any(len(f) != K for _, f in recs) or not recs:
            continue
        po = pacsv.ParseOptions(quote_char=quote, escape_char=escape or False, double_quote=True, newlines_in_values=True)
        co = pacsv.ConvertOptions(column_types={f"c{j}": pa.string() for j in range(K)}, null_values=["NA", "null", "\\N"],
                                  strings_can_be_null=True, quoted_strings_can_be_null=True)
        ro = pacsv.ReadOptions(column_names=[f"c{j}" for j in range(K)])
        got = pacsv.read_csv(io.BytesIO(data), read_options=ro, parse_options=po, convert_options=co)
        for j in range(K):
            want = [None if isn else v.decode() for v, isn in (f[j] for _, f in recs)]
            assert got.column(j).to_pylist() == want, (trial, data, j)


def _random_format(rng):
    while True:
        kw = dict(delimiter=rng.choice([",", ";", "\t"]), quote=rng.choice(['"', "'"]), escape=rng.choice([None, "\\"]),
                  comment=rng.choice([None, "#"]), terminator=rng.choice([None, "\n", ";", "|"]))
        special = [kw[k] for k in ("delimiter", "quote", "escape", "comment", "terminator") if kw[k]]
        if kw["terminator"] is None:
            special += ["\n", "\r"]
        if len(set(special)) == len(special):
            return kw


def test_split_host_equals_the_model_on_fuzzed_inputs(built_lib):
    rng = random.Random(20261021)
    for trial in range(100_000):
        kw = _random_format(rng)
        rx = rng.choice([None, "dump", "empty"])
        alphabet = [kw["delimiter"], kw["quote"], "\\", "#", ";", "|", "\r", "\n", "a", "b", "N", "A"]
        data = "".join(rng.choice(alphabet) for _ in range(rng.randint(0, 40))).encode()
        recs, _, err = model(data, null=NULL_PY[rx], **kw)
        st, got = split_host(data, null_regex=NULL_RX[rx], **kw)
        if err:
            assert st == INVALID_ARG and f"CSV line {err[1]}: unterminated quote" in got, (trial, kw, data, got)
        else:
            assert st == 0 and got == recs, (trial, kw, rx, data, got, recs)


def test_special_byte_clashes_are_refused(built_lib):
    names = ["delimiter", "quote", "escape", "comment", "terminator"]
    for a in range(5):
        for b in range(a + 1, 5):
            kw = dict(delimiter=",", quote='"', escape=None, comment=None, terminator=None)
            kw[names[a]] = kw[names[b]] = "|"
            st, msg = split_host(b"x", **kw)
            assert st == INVALID_ARG and f"the {names[a]} and the {names[b]} are the same byte '|'" in msg, (kw, msg)
    for k in ("delimiter", "quote", "escape", "comment"):  # the default terminator is CR and LF
        for c, what in (("\n", "LF"), ("\r", "CR")):
            st, msg = split_host(b"x", **{k: c})
            assert st == INVALID_ARG and f"the {k} and the terminator ({what})" in msg, (k, msg)
    assert split_host(b"a\nb", delimiter="\n", terminator=";")[0] == 0  # with another terminator LF is an ordinary byte
    with pytest.raises(ValueError):
        fmt_of(escape="ab")


def test_null_regex_errors(built_lib):
    st, msg = split_host(b"x", null_regex="(NA")
    assert st == INVALID_ARG and "NULL regex" in msg, msg
    for rx in (r"(?=NA)", r"(a)\1"):  # no look-around or back-references in the regex crate either
        st, msg = split_host(b"x", null_regex=rx)
        assert st == INVALID_ARG and "NULL regex" in msg, (rx, st, msg)
    st, msg = split_host(b"x", null_regex=r"[ab]*a[ab]{14}")  # more DFA states than the compiler builds
    assert st == F.TG_ERR_UNSUPPORTED and "NULL regex" in msg and "DFA states" in msg, msg
    assert split_host(b"NA,x,\\N\n", null_regex=r"^(NA|\\N|null)$") == (0, [(1, [(b"NA", True), (b"x", False), (b"\\N", True)])])
    assert split_host(b"xNAx,", null_regex="NA") == (0, [(1, [(b"xNAx", True), (b"", False)])])  # unanchored search


def test_dialect_semantics_by_example(built_lib):
    # escape only inside quotes; CRLF read with terminator LF keeps the CR; comments only at a record's start
    assert split_host(b'"a\\"b",c\\d\n', escape="\\")[1] == [(1, [(b'a"b', False), (b"c\\d", False)])]
    assert split_host(b"a,b\r\nc,d\r\n", terminator="\n")[1] == [(1, [(b"a", False), (b"b\r", False)]), (2, [(b"c", False), (b"d\r", False)])]
    assert split_host(b"#x,\"y\n\n\na,#b\n#c\nd", comment="#")[1] == [(4, [(b"a", False), (b"#b", False)]), (6, [(b"d", False)])]
    assert split_host(b"a;;b;", terminator=";")[1] == [(1, [(b"a", False)]), (3, [(b"b", False)])]
    assert split_host(b"'it''s',x", quote="'")[1] == [(1, [(b"it's", False), (b"x", False)])]


# ------------------------------------------------------------------------------------------ GPU ----
NULL_TOKENS = {None: ["", '""'], "dump": ["NA", "\\N", "null", '"NA"'], "empty": ["", "NA", '""']}  # '"': the dialect's quote


def _text(v, k):
    import datetime as dt
    if isinstance(v, bool):
        return ("true", "FALSE", "True", "false")[k % 4] if v else ("false", "False")[k % 2]
    if isinstance(v, float):
        return repr(v)
    if isinstance(v, dt.datetime):
        return v.isoformat(sep="T" if k % 2 else " ")
    if isinstance(v, dt.date):
        return v.isoformat()
    return str(v)


def write_dialect(rows, names, delimiter=",", quote='"', escape=None, comment=None, terminator=None, null_regex=None, seed=0, esc_rate=0.3):
    """a file of `rows` in the dialect: NULLs as the dialect's NULL tokens, quoting where a value needs it (and at random),
    escapes and doubled quotes inside quotes, comment and blank lines between records, CRLF for the default terminator"""
    rng = random.Random(seed)
    eol = terminator or "\r\n"
    specials = {delimiter, quote, "\n", "\r"} | ({terminator} if terminator else set()) | ({escape} if escape else set())
    out = []
    if comment:
        out.append(comment + 'a comment, "with" quotes' + (" \\" if escape else "") + eol)
    out.append(delimiter.join(names) + eol)
    for i, r in enumerate(rows):
        fs = []
        for j, v in enumerate(r):
            if v is None:
                fs.append(rng.choice(NULL_TOKENS[null_regex]).replace('"', quote))
                continue
            s = _text(v, i + j)
            need = any(c in s for c in specials) or (j == 0 and comment and s.startswith(comment))
            if need or rng.random() < 0.2:
                body = []
                for c in s:
                    if c == quote:
                        body.append(escape + c if escape and rng.random() < 0.5 else c + c)
                    elif escape and (c == escape or rng.random() < esc_rate / max(len(s), 1)):
                        body.append(escape + c)
                    else:
                        body.append(c)
                s = quote + "".join(body) + quote
            fs.append(s)
        out.append(delimiter.join(fs) + eol)
        if comment and i % 37 == 3:
            out.append(comment + " skipped" + delimiter + quote + eol)
        if i % 53 == 7:
            out.append(eol)
    return "".join(out).encode()


def expected_table(data, schema, **kw):
    """the reference's parse of a file with a header: every column cast from the model's unescaped values"""
    rx = kw.pop("null_regex", None)
    recs, _, err = model(data, null=NULL_PY[rx], **kw)
    assert err is None
    cols = []
    for j, f in enumerate(schema):
        vals = [None if fs[j][1] else fs[j][0].decode() for _, fs in recs[1:]]
        a = pa.array(vals, type=pa.string())
        if pa.types.is_boolean(f.type):
            a = pc.utf8_lower(a)
        cols.append(a if pa.types.is_string(f.type) else a.cast(f.type))
    return pa.table(cols, schema=schema)


def _register(ctx, name, data, tmp_path, schema=SCHEMA, **kw):
    p = tmp_path / (name + ".csv")
    p.write_bytes(data)
    ctx.register_csv(name, str(p), schema, **kw)


def _edge_kinds(data, states, chunk):
    """which of the positions a chunk of `chunk` bytes cuts at fall inside a comment, right after an escape byte, inside
    quotes and between CR and LF"""
    kinds = set()
    for e in range(chunk, len(data), chunk):
        st = states[e]
        if st in ("cmt", "esc", "quo"):
            kinds.add(st)
        if data[e - 1] == 13 and data[e] == 10:
            kinds.add("crlf")
    return kinds


MATRIX = [(q, e, c, t, rx) for q in ('"', "'") for e in (None, "\\") for c in (None, "#") for t in (None, "\n", ";") for rx in (None, "dump", "empty")]


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [None, 4093])
@pytest.mark.parametrize("quote,escape,comment,terminator,rx", MATRIX)
def test_dialect_matrix_decodes_every_type(ctx, tmp_path, monkeypatch, chunk, quote, escape, comment, terminator, rx):
    kw = dict(quote=quote, escape=escape, comment=comment, terminator=terminator)
    data = write_dialect(_rows(1500, 0.1, 21), SCHEMA.names, null_regex=rx, seed=3, **kw)
    want = expected_table(data, SCHEMA, null_regex=rx, **kw)
    if chunk:
        monkeypatch.setenv("TG_CSV_CHUNK_BYTES", str(chunk))
    _register(ctx, "dm", data, tmp_path, null_regex=NULL_RX[rx], **kw)
    try:
        assert ctx.num_rows("dm") == 1500
        _check_table(ctx, "dm", want)
    finally:
        ctx.deregister_table("dm")


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [5, 7, 11, 13, 2039])
def test_small_chunks_cut_inside_comments_escapes_quotes_and_crlf(ctx, tmp_path, monkeypatch, chunk):
    kw = dict(quote='"', escape="\\", comment="#", terminator=None)
    rows = _rows(300, 0.1, 23)
    rows[17][4] = "long " + 'x,"y"\\\n' * 900  # a record longer than several chunks
    data = write_dialect(rows, SCHEMA.names, null_regex="dump", seed=4, esc_rate=3.0, **kw)
    want = expected_table(data, SCHEMA, null_regex="dump", **kw)
    _, states, _ = model(data, **kw)
    kinds = set()
    for c in (5, 7, 11, 13, 2039):
        kinds |= _edge_kinds(data, states, c)
    assert kinds >= {"cmt", "esc", "quo", "crlf"}, kinds
    monkeypatch.setenv("TG_CSV_CHUNK_BYTES", str(chunk))
    _register(ctx, "sc", data, tmp_path, null_regex=NULL_RX["dump"], **kw)
    try:
        assert ctx.num_rows("sc") == 300
        _check_table(ctx, "sc", want)
    finally:
        ctx.deregister_table("sc")


@pytest.mark.gpu
@pytest.mark.parametrize("delim,eol,header,blank", [(",", "\n", True, False), (";", "\r\n", False, True), ("\t", "\r", True, False)])
def test_default_dialect_equals_tg_table_append_csv(ctx, tmp_path, delim, eol, header, blank):
    from tests.test_csv import _write_csv
    path = tmp_path / "d.csv"
    _write_csv(str(path), _rows(4000, 0.05, 31), delim, eol, header, True, blank)
    data = path.read_bytes()
    names, _ = T.api._strs(SCHEMA.names)
    fmts, _ = T.api._strs([T.api._arrow_format(f.type) for f in SCHEMA])
    bufs = []
    for k, name in enumerate(("old", "new")):
        tab = ctx._create(name)
        rows = C.c_int64()
        if k == 0:
            F.check(F.lib().tg_table_append_csv(tab, names, fmts, len(SCHEMA), data, len(data), ord(delim), int(header), C.byref(rows)))
        else:
            f = fmt_of(delimiter=delim, has_header=header)
            F.check(F.lib().tg_table_append_csv_format(tab, names, fmts, len(SCHEMA), data, len(data), C.byref(f), C.byref(rows)))
        assert rows.value == 4000
        got = []
        for col in SCHEMA.names:
            b, valid, vals, offs = _read(ctx, name, col)
            got.append((b["null_count"], b["dtype"], valid.tobytes(), vals.tobytes(), None if offs is None else offs.tobytes()))
        bufs.append(got)
    try:
        assert bufs[0] == bufs[1]
        assert _suite(ctx, "old") == _suite(ctx, "new")  # pivots and every statistic
    finally:
        ctx.deregister_table("old")
        ctx.deregister_table("new")


ERRORS = [  # (text, dialect, schema, message part)
    ('a,b\n1,"x\\', dict(escape="\\"), [("a", "l"), ("b", "u")], "CSV line 2, column 'b': unterminated quote"),
    ('a,b\n1,"x\\"y\n2,3\n', dict(escape="\\"), [("a", "l"), ("b", "u")], "CSV line 2, column 'b': unterminated quote"),
    ("a,b\n\\N,7\nNA,x7\n", dict(null_regex=r"^(NA|\\N)$"), [("a", "l"), ("b", "l")], "CSV line 3, column 'b': cannot parse 'x7' as Int64"),
    ("a,b\n1,\n", dict(null_regex=r"^NA$"), [("a", "l"), ("b", "l")], "CSV line 2, column 'b': cannot parse '' as Int64"),
    ("#c\n\na,b\n#c\n\n1,2\n#c\n3\n", dict(comment="#"), [("a", "l"), ("b", "l")], "CSV line 8, column 'b': missing"),
    ("#c;;a,b;1,2;#x;;q,2;", dict(comment="#", terminator=";"), [("a", "l"), ("b", "l")], "CSV line 7, column 'a': cannot parse 'q' as Int64"),
    ("a,b\r\n1,2\r\n3,4,5\r\n", dict(terminator="\n"), [("a", "l"), ("b", "u")], "CSV line 3, column 'b': followed by an extra field"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [None, 5, 8, 13])
@pytest.mark.parametrize("k", range(len(ERRORS)))
def test_errors_name_the_line_and_change_nothing(ctx, monkeypatch, k, chunk):
    if chunk:
        monkeypatch.setenv("TG_CSV_CHUNK_BYTES", str(chunk))
    text, dialect, schema, msg = ERRORS[k]
    data = text.encode()
    f = fmt_of(**dialect)
    names, _ = T.api._strs([n for n, _ in schema])
    fmts, _ = T.api._strs([t for _, t in schema])
    tab = ctx._create("fe")
    try:
        good = (dialect.get("terminator") or "\n").join(["a,b", "5,6", ""]).encode()
        F.check(F.lib().tg_table_append_csv_format(tab, names, fmts, 2, good, len(good), C.byref(f), None))
        before = [_read(ctx, "fe", n)[1:] for n, _ in schema]
        st = F.lib().tg_table_append_csv_format(tab, names, fmts, 2, data, len(data), C.byref(f), None)
        assert st == INVALID_ARG and msg in F.last_error(), (st, F.last_error())
        after = [_read(ctx, "fe", n)[1:] for n, _ in schema]
        for (v0, b0, o0), (v1, b1, o1) in zip(before, after):
            assert (v0 == v1).all() and b0.tobytes() == b1.tobytes() and (o0 is None or (o0 == o1).all())
        assert ctx.num_rows("fe") == 1
    finally:
        ctx.deregister_table("fe")


@pytest.mark.gpu
def test_suite_over_a_dump_style_file_equals_the_suite_over_arrow(ctx, tmp_path):
    kw = dict(quote='"', escape="\\", comment="#", terminator=None)
    data = write_dialect(_rows(20000, 0.05, 9), SCHEMA.names, null_regex="dump", seed=5, **kw)
    want = expected_table(data, SCHEMA, null_regex="dump", **kw)
    _register(ctx, "ds_csv", data, tmp_path, null_regex=NULL_RX["dump"], **kw)
    ctx.register_table("ds_arrow", want)
    try:
        got, exp = _suite(ctx, "ds_csv"), _suite(ctx, "ds_arrow")
        assert got[0] == exp[0], [(a, b) for a, b in zip(got[0], exp[0]) if a != b]
        assert got[1] == exp[1] and len(got[1]) >= 2
    finally:
        ctx.deregister_table("ds_csv")
        ctx.deregister_table("ds_arrow")


@pytest.mark.gpu
def test_full_size_dump_style_file(ctx, tmp_path):
    # ~1 GB over several 256 MiB chunks: Int64, Float64, Utf8 with \ escapes in 10 % of the strings, \N NULLs, # comment lines
    n = 20_000_000
    rng = np.random.default_rng(43)
    ids = rng.integers(-10**15, 10**15, n)
    xs = rng.normal(100.0, 15.0, n)
    path = str(tmp_path / "dump.csv")
    schema = pa.schema([pa.field("id", pa.int64()), pa.field("x", pa.float64()), pa.field("email", pa.string())])
    want_s, want_x = [], []
    step = 1_000_000
    with open(path, "w") as f:
        f.write("# dump\nid,x,email\n")
        for lo in range(0, n, step):
            idx = np.arange(lo, min(n, lo + step))
            plain = np.char.add(np.char.add("user", idx.astype(str)), "@example.com")
            esc = idx % 10 == 0
            quoted = np.char.add(np.char.add('"us\\"er', idx.astype(str)), ',x\\\\@example.com"')  # "us\"er<i>,x\\@example.com"
            em = np.where(esc, quoted, plain)
            nul = idx % 101 == 0
            em = np.where(nul, "\\N", em)
            xn = idx % 97 == 0
            xt = np.where(xn, "\\N", np.char.mod("%.17g", xs[idx]))
            lines = np.char.add(np.char.add(np.char.add(np.char.add(ids[idx].astype(str), ","), xt), ","), em)
            f.write("\n".join(lines.tolist()) + "\n# chunk " + str(lo) + ',"x\n')
            want_s.append(pa.array(np.where(esc, np.char.add(np.char.add('us"er', idx.astype(str)), ",x\\@example.com"), plain), mask=nul))
            want_x.append(pa.array(xs[idx], mask=xn))
    assert os.path.getsize(path) > 700 << 20
    want = pa.table([pa.array(ids), pa.chunked_array(want_x), pa.chunked_array(want_s)], schema=schema)
    ctx.register_csv("dump", path, schema, escape="\\", comment="#", null_regex=r"^\\N$")
    try:
        _check_table(ctx, "dump", want)
    finally:
        ctx.deregister_table("dump")
