"""Arrow string columns delivered dictionary-encoded (dictionary<int*, utf8 | large_utf8>) or as utf8_view: the engine
stores the plain Utf8 column of their logical values, decoded on the device. CPU tests: the arrow-rs names of these types
(what has_consistent_data_type's SpecificType compares with). GPU tests: the decoded buffers bit for bit against the Utf8
registration of the same values, one suite's results on an encoded column against its plain twin and the oracle, the
refused encodings and the malformed-input errors, and a C3-sized dictionary column."""
import numpy as np
import pyarrow as pa
import pyarrow.compute as pc
import pytest

import term_b200 as T
from term_b200 import _ffi as F
from term_b200.api import arrow_type_debug

TG_ERR_INVALID_ARG = next(k for k, v in F.STATUS_NAMES.items() if v == "TG_ERR_INVALID_ARG")

INDEX_TYPES = [(pa.int8(), "Int8"), (pa.uint8(), "UInt8"), (pa.int16(), "Int16"), (pa.uint16(), "UInt16"), (pa.int32(), "Int32"),
               (pa.uint32(), "UInt32"), (pa.int64(), "Int64"), (pa.uint64(), "UInt64")]
VALUE_TYPES = [(pa.string(), "Utf8"), (pa.large_string(), "LargeUtf8")]


@pytest.mark.parametrize("index_type,index_name", INDEX_TYPES)
@pytest.mark.parametrize("value_type,value_name", VALUE_TYPES)
def test_arrow_type_debug_of_string_dictionaries(index_type, index_name, value_type, value_name):
    assert arrow_type_debug(pa.dictionary(index_type, value_type)) == f"Dictionary({index_name}, {value_name})"


def test_arrow_type_debug_of_views():
    assert arrow_type_debug(pa.string_view()) == "Utf8View"
    assert arrow_type_debug(pa.binary_view()) == "BinaryView"


# ------------------------------------------------------------------------------------------ data ----
def _vocab(rng, k):
    """k distinct strings: ASCII, multi-byte UTF-8, the empty string, lengths around the 12-byte view inline limit and far
    above it, e-mail and SSN shapes"""
    fixed = ["", "a", "héllo wörld", "日本語テキスト", "emoji 🎉🎉", "x" * 11, "y" * 12, "z" * 13, "ab" * 40, "long " * 60,
             "user@example.com", "jane.doe@mail.example.org", "not-an-email@", "123-45-6789", "987-65-4321", "abc-de-fghi"]
    out = list(fixed)
    while len(out) < k:
        i = len(out)
        kind = i % 4
        if kind == 0:
            out.append(f"user{i}@host{i % 7}.com")
        elif kind == 1:
            out.append(f"{100 + i % 900:03d}-{10 + i % 90:02d}-{1000 + i:04d}")
        elif kind == 2:
            out.append("v" + "é" * (i % 9) + str(i))
        else:
            out.append(f"value_{i}_" + "q" * (i % 37))
    return out[:k]


def _column(n, k=100, null_p=0.05, seed=3):
    """(dictionary values list, int64 codes, row validity) of one seeded column"""
    rng = np.random.default_rng(seed)
    vocab = _vocab(rng, k)
    codes = rng.integers(0, k, n)
    valid = rng.random(n) >= null_p
    return vocab, codes, valid


def _plain(vocab, codes, valid):
    return pa.array([vocab[c] if ok else None for c, ok in zip(codes, valid)], type=pa.string())


def _dict(vocab, codes, valid, index_type, value_type, perm_seed=None):
    """the same logical column as a dictionary array; perm_seed: the dictionary's order is shuffled (a different dictionary)"""
    order = np.arange(len(vocab))
    if perm_seed is not None:
        order = np.random.default_rng(perm_seed).permutation(len(vocab))
    pos = np.empty_like(order)
    pos[order] = np.arange(len(vocab))
    dictionary = pa.array([vocab[i] for i in order], type=value_type)
    idx = pa.array(pos[codes], mask=~valid).cast(index_type)
    return pa.DictionaryArray.from_arrays(idx, dictionary)


def _view(vocab, codes, valid, pieces=3):
    """utf8_view with several data buffers (one per concatenated piece)"""
    plain = _plain(vocab, codes, valid)
    cuts = np.linspace(0, len(plain), pieces + 1).astype(int)
    arr = pa.concat_arrays([plain.slice(a, b - a).cast(pa.string_view()) for a, b in zip(cuts[:-1], cuts[1:])])
    return arr


# ------------------------------------------------------------------------------------------ GPU ----
def _read_utf8(ctx, table, column):
    """(offsets, bytes, validity, null_count) of a stored Utf8 column, read back from HBM"""
    import torch
    from term_b200.distributed import _tensor_from_ptr
    b = ctx.column_buffers(table, column)
    dev = torch.device("cuda", 0)
    n = b["n_rows"]
    offs = _tensor_from_ptr(b["offsets"], (n + 1) * 4, dev, "|u1").cpu().numpy().view(np.int32).copy()
    data = _tensor_from_ptr(b["values"], max(int(offs[-1]), 1), dev, "|u1").cpu().numpy()[: int(offs[-1])].tobytes()
    if b["validity"]:
        bits = _tensor_from_ptr(b["validity"], (n + 7) // 8, dev, "|u1").cpu().numpy()
        valid = np.unpackbits(bits, bitorder="little")[:n].astype(bool)
    else:
        valid = np.ones(n, dtype=bool)
    assert b["n_value_bytes"] == int(offs[-1])
    return offs, data, valid, int(b["null_count"])


def _assert_same_as_plain(ctx, name, batches, want):
    """register `batches` (column "s") and the Utf8 cast of `want`; every buffer must be equal"""
    ctx.register_table(name, batches)
    ctx.register_table(name + "_ref", pa.table({"s": pc.cast(want, pa.string())}))
    try:
        assert ctx.column_dtype(name, "s") == F.TG_UTF8
        got, ref = _read_utf8(ctx, name, "s"), _read_utf8(ctx, name + "_ref", "s")
        assert (got[0] == ref[0]).all(), name
        assert got[1] == ref[1], name
        assert (got[2] == ref[2]).all(), name
        assert got[3] == ref[3] == int((~ref[2]).sum()), name
    finally:
        ctx.deregister_table(name)
        ctx.deregister_table(name + "_ref")


N = 70_001  # not a multiple of the 1024-row block nor of 8


@pytest.mark.gpu
@pytest.mark.parametrize("value_type", [pa.string(), pa.large_string()], ids=["utf8", "large_utf8"])
@pytest.mark.parametrize("index_type", [t for t, _ in INDEX_TYPES], ids=[nm for _, nm in INDEX_TYPES])
def test_dictionary_decodes_to_the_utf8_buffers(ctx, index_type, value_type):
    vocab, codes, valid = _column(N)
    arr = _dict(vocab, codes, valid, index_type, value_type)
    _assert_same_as_plain(ctx, "enc_dict", pa.table({"s": arr}), arr)


@pytest.mark.gpu
def test_dictionary_with_null_values_is_a_logical_null(ctx):
    vocab, codes, valid = _column(N, seed=5)
    dictionary = pa.array([None if i % 10 == 3 else v for i, v in enumerate(vocab)], type=pa.string())
    arr = pa.DictionaryArray.from_arrays(pa.array(codes.astype(np.int16), mask=~valid), dictionary)
    want = pc.cast(arr, pa.string())
    assert want.null_count > arr.null_count  # some valid rows name a NULL value
    _assert_same_as_plain(ctx, "enc_dnull", pa.table({"s": arr}), arr)


@pytest.mark.gpu
def test_view_with_several_data_buffers_decodes_to_the_utf8_buffers(ctx):
    vocab, codes, valid = _column(N, seed=7)
    arr = _view(vocab, codes, valid)
    assert len(arr.buffers()) >= 5  # validity, views, three data buffers
    _assert_same_as_plain(ctx, "enc_view", pa.table({"s": arr}), arr)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["dict", "large_dict", "view"])
def test_sliced_batches(ctx, kind):
    vocab, codes, valid = _column(N, seed=9)
    arr = {"dict": lambda: _dict(vocab, codes, valid, pa.int32(), pa.string()),
           "large_dict": lambda: _dict(vocab, codes, valid, pa.uint8(), pa.large_string()),
           "view": lambda: _view(vocab, codes, valid)}[kind]()
    # the dictionary child sliced too: its offset is not zero
    if kind == "dict":
        arr = pa.DictionaryArray.from_arrays(arr.indices, pa.concat_arrays([pa.array(["pad0", "pad1"]), arr.dictionary]).slice(2))
    cuts = [0, 3, 1027, 5000, 5001, 40_000, N]
    batches = [pa.record_batch([arr.slice(a, b - a)], names=["s"]) for a, b in zip(cuts[:-1], cuts[1:])]
    assert any(b.column(0).offset % 8 for b in batches)
    _assert_same_as_plain(ctx, "enc_slice", batches, arr)


@pytest.mark.gpu
def test_one_column_mixing_encodings_and_dictionaries(ctx):
    vocab, codes, valid = _column(N, seed=11)
    cuts = [0, 999, 12_345, 20_000, 33_333, 50_001, 61_000, N]
    parts = []
    for k, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])):
        c, v = codes[a:b], valid[a:b]
        parts.append([lambda: _plain(vocab, c, v),
                      lambda: _dict(vocab, c, v, pa.int8(), pa.string(), perm_seed=k),
                      lambda: _view(vocab, c, v, pieces=2),
                      lambda: _dict(vocab, c, v, pa.uint32(), pa.large_string(), perm_seed=100 + k),
                      lambda: _plain(vocab, c, v).cast(pa.large_string()),
                      lambda: _dict(vocab, c, v, pa.int64(), pa.string()).slice(0),
                      lambda: _view(vocab, c, v, pieces=1)][k]())
    batches = [pa.record_batch([p], names=["s"]) for p in parts]
    _assert_same_as_plain(ctx, "enc_mix", batches, _plain(vocab, codes, valid))


def _suite(col, parent):
    hist = lambda h: h.most_common_ratio() < 0.5  # noqa: E731
    return (T.Check.builder("enc")
            .completeness(col, 0.9)
            .validates_uniqueness([col], 0.1)
            .validates_distinctness([col], T.Assertion.GreaterThan(0.0))
            .has_approx_count_distinct(col, T.Assertion.GreaterThan(10.0))
            .validates_email(col, 0.1)
            .contains_ssn(col, 0.05)
            .validates_regex(col, r"^[a-z]+[0-9]", 0.1)
            .has_min_length(col, 1)
            .has_max_length(col, 100)
            .has_length_between(col, 2, 40)
            .satisfies(f"{col} = 'user@example.com'")
            .satisfies(f"{col} < 'm'")
            .satisfies(f"{col} LIKE 'user%'")
            .satisfies(f"LENGTH({col}) > 12")
            .has_histogram_with_description(col, hist, "no dominant value")
            .foreign_key(f"data_enc.{col}", f"{parent}.p")
            .build())


def _oracle(t, tables, col):
    from oracle import term_oracle as O
    return [O.completeness(t, col, 0.9), O.uniqueness(t, [col], "FullUniqueness", 0.1),
            O.uniqueness(t, [col], "Distinctness", assertion=("GreaterThan", 0.0)), None,
            O.format_constraint(t, col, "Email", 0.1), O.format_constraint(t, col, "SocialSecurityNumber", 0.05, trim=True),
            O.format_constraint(t, col, "Regex", 0.1, arg=r"^[a-z]+[0-9]"),
            O.length_constraint(t, col, "Min", 1), O.length_constraint(t, col, "Max", 100), O.length_constraint(t, col, "Between", 2, 40),
            O.custom_sql(t, f"{col} = 'user@example.com'"), O.custom_sql(t, f"{col} < 'm'"), O.custom_sql(t, f"{col} LIKE 'user%'"),
            O.custom_sql(t, f"LENGTH({col}) > 12"),
            O.histogram_constraint(t, col, lambda h: h.most_common_ratio() < 0.5, "no dominant value"),
            O.foreign_key(tables, f"data_enc.{col}", "parent.p")[0]]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["dict", "view"])
def test_suite_on_an_encoded_column_equals_its_plain_twin_and_the_oracle(ctx, kind):
    n = 120_007
    vocab, codes, valid = _column(n, k=400, seed=13)
    enc = _dict(vocab, codes, valid, pa.int32(), pa.string()) if kind == "dict" else _view(vocab, codes, valid)
    plain = _plain(vocab, codes, valid)
    t = pa.table({"s_enc": enc, "s_plain": plain, "v": pa.array(np.arange(n, dtype=np.float64), mask=np.arange(n) % 7 == 0)})
    parent = pa.table({"p": pa.array(vocab[::2], type=pa.string())})
    ctx.register_table("data_enc", t.to_batches(max_chunksize=50_000))
    ctx.register_table("parent", parent)
    try:
        res = {}
        for col in ("s_enc", "s_plain"):
            res[col] = T.ValidationSuite.builder("enc").table_name("data_enc").check(_suite(col, "parent")).build().run(ctx).report.results
        decoded = pa.table({"s_enc": pc.cast(enc, pa.string()), "s_plain": plain, "v": t.column("v")})
        want = _oracle(decoded, {"data_enc": decoded, "parent": parent}, "s_plain")
        assert len(res["s_enc"]) == len(want)
        def msg(r):  # which foreign-key example values are listed is unpinned (DESIGN §5): the message up to them
            m = (r.message or "").replace("s_enc", "s_plain")
            return m.split(" Examples:")[0].rstrip(".") if r.name == "foreign_key" else m

        for g, p, w in zip(res["s_enc"], res["s_plain"], want):
            assert g.status == p.status and g.metric == p.metric and msg(g) == msg(p), (g, p)
            if w is None:  # approx_count_distinct: HyperLogLog, the oracle's count is exact
                continue
            w.name = p.name
            assert p.status.name.lower() == w.status and msg(p) == msg(w), (p, w)
            if w.metric is None or p.metric is None:
                assert w.metric is None and p.metric is None, (p, w)
            else:  # (the histogram's entropy is a float sum: its order may differ from the oracle's)
                assert p.metric == pytest.approx(w.metric, rel=1e-9, abs=1e-12), (p, w)
        # grouped completeness grouped by the encoded column
        from oracle import term_oracle as O
        maps = []
        for col in ("s_enc", "s_plain"):
            plan = T.Plan()
            slot = T.GroupedCompletenessAnalyzer("v", [col])._add_to(plan)
            plan.execute(ctx, "data_enc")
            maps.append(plan.analyzer_result(slot).map)
        assert maps[0] == maps[1]
        og = O.grouped_completeness(decoded, "v", ["s_plain"])
        assert {k: v for k, v in maps[0].items() if not k.startswith("__")} == \
               {"NULL" if k[0] is None else str(k[0]): nn / tt for k, (tt, nn) in og.items()}
        # the schema keeps the delivered type: SpecificType matches arrow-rs's name of it
        want_type = "Dictionary(Int32, Utf8)" if kind == "dict" else "Utf8View"
        U = T.UnifiedDataTypeConstraint
        rs = T.ValidationSuite.builder("t").table_name("data_enc").check(
            T.Check.builder("t").constraint(U.specific_type("s_enc", want_type)).constraint(U.specific_type("s_enc", "Utf8")).build()
        ).build().run(ctx).report.results
        assert rs[0].status.name == "Success" and rs[1].status.name == "Failure", rs
    finally:
        ctx.deregister_table("data_enc")
        ctx.deregister_table("parent")


def _register_fails(ctx, name, table):
    with pytest.raises(T.TermGpuError) as ei:
        ctx.register_table(name, table)
    with pytest.raises(T.TermGpuError):
        ctx.num_rows(name)  # the failed registration left no table behind
    return ei.value


@pytest.mark.gpu
def test_refused_encodings(ctx):
    bv = pa.array([b"abc", None, b"a much longer binary value"], type=pa.binary_view())
    bdict = pa.array([b"x", b"y", b"x"], type=pa.binary()).dictionary_encode()
    idict = pa.array([1, 2, 1, 5], type=pa.int64()).dictionary_encode()
    for name, arr, what in (("r_bv", bv, "BinaryView"), ("r_bd", bdict, "Binary"), ("r_id", idict, "Int64")):
        err = _register_fails(ctx, name, pa.table({"ok": pa.array(["a"] * len(arr)), "s": arr}))
        assert err.code == F.TG_ERR_UNSUPPORTED and what in str(err), (name, err)


@pytest.mark.gpu
def test_malformed_input_is_an_error(ctx):
    # a valid row whose index lies outside the dictionary (its NULL rows carry an out-of-range index too: never read)
    idx = pa.array([0, 1, 7, None, 2], type=pa.int32())
    bad = pa.DictionaryArray.from_arrays(idx, pa.array(["a", "b", "c"]), safe=False)
    err = _register_fails(ctx, "m_idx", pa.table({"s": bad}))
    assert err.code == TG_ERR_INVALID_ARG and "outside the dictionary" in str(err)
    # the same with an empty dictionary
    empty = pa.DictionaryArray.from_arrays(pa.array([0, None], type=pa.int8()), pa.array([], type=pa.string()), safe=False)
    assert _register_fails(ctx, "m_empty", pa.table({"s": empty})).code == TG_ERR_INVALID_ARG
    # an index under a NULL row is undefined in Arrow: not an error
    ok = pa.DictionaryArray.from_arrays(pa.array([0, 99, 1], type=pa.int8(), mask=np.array([False, True, False])), pa.array(["a", "b"]), safe=False)
    ctx.register_table("m_ok", pa.table({"s": ok}))
    try:
        assert ctx.num_rows("m_ok") == 3 and _read_utf8(ctx, "m_ok", "s")[3] == 1
    finally:
        ctx.deregister_table("m_ok")
    # a view whose offset + length lies past its data buffer
    good = pa.array(["short", "a value longer than twelve bytes"], type=pa.string_view())
    views = np.frombuffer(good.buffers()[1], dtype=np.uint32).copy().reshape(-1, 4)
    views[1, 3] += 10  # offset of the long value moved past the end of its 32-byte buffer
    forged = pa.Array.from_buffers(pa.string_view(), 2, [None, pa.py_buffer(views.tobytes()), good.buffers()[2]])
    err = _register_fails(ctx, "m_view", pa.table({"s": forged}))
    assert err.code == TG_ERR_INVALID_ARG and "outside its data buffer" in str(err)


@pytest.mark.gpu
def test_c3_sized_dictionary_column_gives_the_plain_results(ctx):
    """25 M rows, about 24 B per value, 1 000 distinct values: the C3 suite on dictionary<int32, utf8> and on Utf8"""
    n = 25_000_000
    rng = np.random.default_rng(17)
    vocab = []
    for i in range(1000):
        L = int(np.clip(rng.poisson(24), 8, 64))
        if i % 10 < 7:
            base = f"u{i}@ex{i % 13}.com"
        elif i % 10 == 7:
            base = f"{100 + i % 800:03d}-{10 + i % 89:02d}-{1000 + i:04d}"
        else:
            base = f"free text {i} "
        vocab.append((base + "x" * max(0, L - len(base)))[:max(L, len(base))])
    codes = rng.integers(0, 1000, n).astype(np.int32)
    valid = rng.random(n) >= 0.02
    enc = pa.DictionaryArray.from_arrays(pa.array(codes, mask=~valid), pa.array(vocab, type=pa.string()))
    plain = pc.cast(enc, pa.string())
    check = lambda: (T.Check.builder("pii").validates_regex("s", "@", 0.5).validates_email("s", 0.5).contains_ssn("s", 0.05)  # noqa: E731
                     .validates_credit_card("s", 0.5, True).build())
    out = []
    for name, arr in (("c3_dict", enc), ("c3_plain", plain)):
        ctx.register_table(name, pa.table({"s": arr}))
        try:
            rs = T.ValidationSuite.builder("c3").table_name(name).check(check()).build().run(ctx).report.results
            out.append([(r.name, r.status, r.metric, r.message) for r in rs])
        finally:
            ctx.deregister_table(name)
    assert out[0] == out[1]
    assert 0.6 < out[0][1][2] < 0.8  # e-mail share: 70 % of the dictionary values are e-mail shaped
