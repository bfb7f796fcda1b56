"""Row verdicts on the GPU (tg_plan_request_row_mask / tg_plan_export_row_mask): the exported Arrow Boolean arrays are
bit-exact against the reference masks built from the oracle's row evaluation, their popcounts reproduce the plan's own
metric, and requesting them changes no result."""
import ctypes as C

import numpy as np
import pyarrow as pa
import pytest

import term_b200 as T
from term_b200 import _ffi as F
from tests import row_mask_reference as R

pytestmark = pytest.mark.gpu
TG_ERR_INVALID_ARG = 1
TILE = 4096


def _drop(ctx, name):
    try:
        ctx.deregister_table(name)
    except T.TermGpuError:
        pass


def _register(ctx, name, table):
    _drop(ctx, name)
    ctx.register_table(name, table)


def _strs(*a):
    return (C.c_char_p * len(a))(*[s.encode() for s in a])


def _read(m):
    import torch
    from term_b200.distributed import _tensor_from_ptr
    n, dev = m.length, torch.device("cuda", 0)
    nb = max((n + 7) // 8, 1)

    def bits(ptr):
        raw = _tensor_from_ptr(ptr, nb, dev, "|u1").cpu().numpy()[:nb].copy()
        return R.unpack(raw.tobytes(), n), raw

    vals, vraw = bits(m.values_ptr)
    if n % 8:
        assert vraw[-1] >> (n % 8) == 0, "bits past n_rows are set"
    if m.validity_ptr:
        valid, _ = bits(m.validity_ptr)
    else:
        valid = np.ones(n, dtype=bool)
    assert m.null_count == int(n - valid.sum())
    return vals, valid


WORDS = ["user@example.com", "bad.example.com", "12", "-7", "x", "", "héllo wörld", "日本語テキスト", "  a@b.co  ", "A@B.COM", "3.5"]


def _table(n, null_p, seed=1):
    rng = np.random.default_rng(seed)
    def mask():
        if null_p == 0:
            return None
        return np.ones(n, dtype=bool) if null_p == 1.0 else rng.random(n) < null_p
    return pa.table({
        "a": pa.array(rng.integers(-5, 10, n), type=pa.int64(), mask=mask()),
        "f": pa.array(rng.normal(1.0, 2.0, n), mask=mask()),
        "i32": pa.array(rng.integers(-100, 100, n).astype(np.int32), mask=mask()),
        "bo": pa.array(rng.random(n) < 0.5, mask=mask()),
        "s": pa.array([WORDS[k] for k in rng.integers(0, len(WORDS), n)], type=pa.string(), mask=mask()),
        "d": pa.array(rng.integers(17000, 20000, n).astype(np.int32), mask=mask()).view(pa.date32()),
    })


def _slots(p):
    """(name, slot, reference(table)) of every row-level kind"""
    lib = F.lib()
    h = p.handle
    O = R.O
    email = O.format_pattern("Email")
    fo = lambda cs, tr, niv: C.byref(F.tg_format_options(cs, tr, niv))
    out = [
        ("completeness", lib.tg_plan_add_completeness(h, _strs("a"), 1, 1.0, 0, 0), lambda t: R.completeness_mask(t, "a")),
        ("completeness_s", lib.tg_plan_add_completeness(h, _strs("s"), 1, 1.0, 0, 0), lambda t: R.completeness_mask(t, "s")),
        ("terms", lib.tg_plan_add_custom_sql(h, b"a > 3 AND f IS NOT NULL", None), lambda t: R.predicate_mask(t, "a > 3 AND f IS NOT NULL")),
        ("terms_or", lib.tg_plan_add_custom_sql(h, b"i32 < 0 OR bo IS NULL", None), lambda t: R.predicate_mask(t, "i32 < 0 OR bo IS NULL")),
        ("arith", lib.tg_plan_add_custom_sql(h, b"(a + i32) * 2 > f OR bo", None), lambda t: R.predicate_mask(t, "(a + i32) * 2 > f OR bo")),
        ("case", lib.tg_plan_add_custom_sql(h, b"CASE WHEN a > 0 THEN f ELSE -f END > 0.5", None),
         lambda t: R.predicate_mask(t, "CASE WHEN a > 0 THEN f ELSE -f END > 0.5")),
        ("coalesce", lib.tg_plan_add_custom_sql(h, b"COALESCE(f, 0.0) > 1.0", None), lambda t: R.predicate_mask(t, "COALESCE(f, 0.0) > 1.0")),
        ("like", lib.tg_plan_add_custom_sql(h, b"s LIKE 'user%' OR s = 'x'", None), lambda t: R.predicate_mask(t, "s LIKE 'user%' OR s = 'x'")),
        ("date", lib.tg_plan_add_custom_sql(h, b"d >= DATE '2019-01-01'", None), lambda t: R.predicate_mask(t, "d >= DATE '2019-01-01'")),
        ("compliance", lib.tg_plan_add_analyzer(h, 13, None, None, b"a >= 0"), lambda t: R.predicate_mask(t, "a >= 0")),
        ("an_completeness", lib.tg_plan_add_analyzer(h, 1, b"f", None, None), lambda t: R.completeness_mask(t, "f")),
        ("containment", lib.tg_plan_add_containment(h, b"s", _strs("x", "12", "日本語テキスト"), 3),
         lambda t: R.containment_mask(t, "s", ["x", "12", "日本語テキスト"])),
        ("non_negative", lib.tg_plan_add_non_negative(h, b"f"), lambda t: R.non_negative_mask(t, "f")),
        ("non_negative_i32", lib.tg_plan_add_non_negative(h, b"i32"), lambda t: R.non_negative_mask(t, "i32")),
        # two slots on one aggregate, null_is_valid true and false
        ("email_niv", lib.tg_plan_add_format(h, b"s", 1, None, 0, 0.5, fo(1, 0, 1)), lambda t: R.format_mask(t, "s", email, True, False, True)),
        ("email_strict", lib.tg_plan_add_format(h, b"s", 1, None, 0, 0.5, fo(1, 0, 0)), lambda t: R.format_mask(t, "s", email, True, False, False)),
        ("email_trim_ci", lib.tg_plan_add_format(h, b"s", 0, b"^[a-z]@[a-z]\\.co$", 0, 0.5, fo(0, 1, 1)),
         lambda t: R.format_mask(t, "s", "^[a-z]@[a-z]\\.co$", False, True, True)),
        ("regex_at", lib.tg_plan_add_format(h, b"s", 0, b"@", 0, 0.5, fo(1, 0, 0)), lambda t: R.format_mask(t, "s", "@", True, False, False)),
        ("data_type", lib.tg_plan_add_data_type(h, b"s", 0, 0.5), lambda t: R.data_type_mask(t, "s", "Integer")),
        ("len_min", lib.tg_plan_add_length(h, b"s", 0, 3, 0), lambda t: R.length_mask(t, "s", 3)),
        ("len_between", lib.tg_plan_add_length(h, b"s", 2, 2, 7), lambda t: R.length_mask(t, "s", 2, 7)),
        ("len_exact", lib.tg_plan_add_length(h, b"s", 3, 7, 0), lambda t: R.length_mask(t, "s", 7, 7)),
    ]
    assert all(s >= 0 for _, s, _ in out), [(n, s) for n, s, _ in out]
    return out


def _plan_with_masks(ctx, request=True, table="data"):
    p = T.api.Plan()
    slots = _slots(p)
    if request:
        for _, s, _ in slots:
            p.request_row_mask(s)
    return p, slots


def _identity(p, slot, vals, valid):
    r = p.result(slot)
    den = int(valid.sum())
    if r.metric is None:
        return
    assert den > 0
    assert float(int((vals & valid).sum())) / float(den) == r.metric


@pytest.mark.parametrize("n", [0, 1, 31, 33, TILE + 5])
@pytest.mark.parametrize("null_p", [0.0, 0.05, 1.0])
def test_bit_exact_against_the_oracle(ctx, n, null_p):
    t = _table(n, null_p, seed=n + int(null_p * 100))
    _register(ctx, "rm_data", t)
    p, slots = _plan_with_masks(ctx)
    p.execute(ctx, "rm_data")
    for name, s, ref in slots:
        m = p.row_mask(s)
        assert m.length == n
        vals, valid = _read(m)
        want_v, want_ok = (np.array(x, dtype=bool).reshape(-1) for x in ref(t))
        assert np.array_equal(valid, want_ok), name
        assert np.array_equal(vals & valid, want_v & want_ok), name
        _identity(p, s, vals, valid)


def test_results_unchanged_by_requests(ctx):
    t = _table(TILE * 3 + 77, 0.05, seed=5)
    _register(ctx, "rm_data", t)
    a, sa = _plan_with_masks(ctx, request=True)
    b, sb = _plan_with_masks(ctx, request=False)
    a.execute(ctx, "rm_data")
    b.execute(ctx, "rm_data")
    for (name, s, _), (_, s2, _) in zip(sa, sb):
        ra, rb = a.result(s), b.result(s2)
        assert (ra.status, ra.metric, ra.message) == (rb.status, rb.metric, rb.message), name


def test_three_million_rows_popcount_identity(ctx):
    n = 3_000_017
    rng = np.random.default_rng(3)
    a = rng.integers(-5, 10, n)
    fv = rng.normal(1.0, 2.0, n)
    fnull = rng.random(n) < 0.05
    words = np.array(WORDS, dtype=object)[rng.integers(0, len(WORDS), n)]
    t = pa.table({"a": pa.array(a), "f": pa.array(fv, mask=fnull), "i32": pa.array(a.astype(np.int32)),
                  "bo": pa.array(a > 2), "s": pa.array(list(words), type=pa.string()),
                  "d": pa.array(np.full(n, 18000, dtype=np.int32)).view(pa.date32())})
    _register(ctx, "rm_data", t)
    p, slots = _plan_with_masks(ctx)
    p.execute(ctx, "rm_data")
    by = {name: s for name, s, _ in slots}
    for name, s, _ in slots:
        vals, valid = _read(p.row_mask(s))
        _identity(p, s, vals, valid)
    vals, _ = _read(p.row_mask(by["terms"]))
    assert np.array_equal(vals, (a > 3) & ~fnull)
    vals, valid = _read(p.row_mask(by["non_negative"]))
    assert np.array_equal(valid, ~fnull) and np.array_equal(vals & valid, (fv >= 0) & ~fnull)
    lens = np.array([len(w) for w in words])
    vals, _ = _read(p.row_mask(by["len_between"]))
    assert np.array_equal(vals, (lens >= 2) & (lens <= 7))
    # two rows per lane in the DFA kernel at this size
    for name, pat in (("regex_at", "@"), ("email_niv", R.O.format_pattern("Email"))):
        per_word = {w: R.format_mask(pa.table({"s": pa.array([w])}), "s", pat)[0][0] for w in WORDS}
        vals, _ = _read(p.row_mask(by[name]))
        assert np.array_equal(vals, np.array([per_word[w] for w in words])), name


@pytest.mark.parametrize("units", [None, "40"])
def test_both_state_layouts(ctx, monkeypatch, units):
    """20 masked predicates next to unmasked aggregates; with 40 units per pass the per-lane state lives in shared memory"""
    if units:
        monkeypatch.setenv("TG_SCAN_UNITS", units)
    n = TILE * 5 + 99
    rng = np.random.default_rng(11)
    a, b = rng.integers(-50, 50, n), rng.normal(0, 10, n)
    bnull = rng.random(n) < 0.1
    t = pa.table({"a": pa.array(a), "b": pa.array(b, mask=bnull)})
    _register(ctx, "rm_data", t)
    p = T.api.Plan()
    lib = F.lib()
    preds = [f"a > {k - 10}" if k % 2 else f"a * 2 + {k} > b" for k in range(20)]
    slots = [lib.tg_plan_add_custom_sql(p.handle, e.encode(), None) for e in preds]
    A = F.tg_assertion(0, 0.0, 0.0)
    for st in range(5):
        lib.tg_plan_add_statistic(p.handle, b"b", st, 0.0, A)
    for s in slots:
        p.request_row_mask(s)
    p.execute(ctx, "rm_data")
    assert p.stats()["scan_smem_state"] == (1 if units else 0)
    for e, s in zip(preds, slots):
        vals, valid = _read(p.row_mask(s))
        want = (a > int(e.split()[-1])) if e.startswith("a >") else ((a * 2 + int(e.split()[4]) > b) & ~bnull)
        assert np.array_equal(vals, want), e
        _identity(p, s, vals, valid)


@pytest.mark.parametrize("env", [{}, {"TG_STR_NO_DIRECT": "1"}])
def test_dfa_variants(ctx, monkeypatch, env):
    """several patterns in one product, long strings past the warp stage, both block shapes / table layouts"""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    n = 20_000
    rng = np.random.default_rng(21)
    pool = WORDS + ["q" * 9000 + "@x.io", "long " * 500, "123-45-6789", "4111 1111 1111 1111"]
    col = [pool[k] if rng.random() > 0.03 else None for k in rng.integers(0, len(pool), n)]
    t = pa.table({"s": pa.array(col, type=pa.string())})
    _register(ctx, "rm_data", t)
    p = T.api.Plan()
    lib = F.lib()
    O = R.O
    specs = [("Email", None), ("SocialSecurityNumber", None), ("CreditCard", None), ("Regex", "@"), ("Regex", "^[0-9]+$"), ("Regex", "o"),
             ("Regex", "l{2}"), ("Regex", "^x$"), ("Regex", "q+@"), ("UUID", None)]
    kinds = {"Regex": 0, "Email": 1, "CreditCard": 3, "UUID": 6, "SocialSecurityNumber": 11}
    slots = []
    for kind, arg in specs:
        s = lib.tg_plan_add_format(p.handle, b"s", kinds[kind], arg.encode() if arg else None, 0, 0.5, None)
        p.request_row_mask(s)
        slots.append((s, O.format_pattern(kind, arg)))
    p.execute(ctx, "rm_data")
    for s, pat in slots:
        vals, valid = _read(p.row_mask(s))
        want, _ = R.format_mask(t, "s", pat)
        assert np.array_equal(vals, np.array(want)), pat
        _identity(p, s, vals, valid)


def test_lifetime_and_errors(ctx):
    t = _table(1000, 0.05, seed=9)
    _register(ctx, "rm_data", t)
    p = T.api.Plan()
    lib = F.lib()
    s = lib.tg_plan_add_custom_sql(p.handle, b"a > 3", None)
    div0 = lib.tg_plan_add_custom_sql(p.handle, b"a / (a - a) > 1", None)
    missing = lib.tg_plan_add_custom_sql(p.handle, b"nope > 1", None)
    badtype = lib.tg_plan_add_format(p.handle, b"a", 1, None, 0, 1.0, None)
    unreq = lib.tg_plan_add_custom_sql(p.handle, b"a > 4", None)
    for x in (s, div0, missing, badtype):
        p.request_row_mask(x)
    p.execute(ctx, "rm_data")
    old = p.row_mask(s)
    old_vals, _ = _read(old)
    for x, code in ((div0, TG_ERR_INVALID_ARG), (missing, 2), (badtype, 3), (unreq, TG_ERR_INVALID_ARG)):
        with pytest.raises(T.TermGpuError) as e:
            p.row_mask(x)
        assert e.value.code == code, (x, e.value)
    # re-execute after an append: the old array keeps its length and bits
    h = C.c_void_p()
    F.check(F.lib().tg_table_lookup(ctx.handle, b"rm_data", C.byref(h)))
    for b in _table(500, 0.05, seed=10).to_batches():
        ctx._append_batch(h, b, False)
    p.execute(ctx, "rm_data")
    new = p.row_mask(s)
    assert new.length == 1500 and old.length == 1000
    assert np.array_equal(_read(old)[0], old_vals)
    assert np.array_equal(_read(new)[0][:1000], old_vals)
    # a request after the last execute makes the mask unavailable until the next one
    p.request_row_mask(unreq)
    with pytest.raises(T.TermGpuError):
        p.row_mask(unreq)
    del p
    import gc
    gc.collect()
    assert np.array_equal(_read(old)[0], old_vals)  # survives the plan


def test_partial_shards_concatenate(ctx):
    t = _table(3 * TILE + 1234, 0.05, seed=4)
    cuts = [0, 1000, 1000 + TILE + 7, t.num_rows]
    p_full, sl = _plan_with_masks(ctx)
    _register(ctx, "rm_data", t)
    p_full.execute(ctx, "rm_data")
    full = {name: _read(p_full.row_mask(s)) for name, s, _ in sl}
    parts = {name: ([], []) for name, _, _ in sl}
    for i in range(3):
        _register(ctx, f"rm_shard{i}", t.slice(cuts[i], cuts[i + 1] - cuts[i]))
        p, sl2 = _plan_with_masks(ctx)
        p.execute_partial(ctx, f"rm_shard{i}")
        for name, s, _ in sl2:
            v, ok = _read(p.row_mask(s))
            parts[name][0].append(v)
            parts[name][1].append(ok)
    for name in full:
        assert np.array_equal(np.concatenate(parts[name][0]) & np.concatenate(parts[name][1]), full[name][0] & full[name][1]), name
        assert np.array_equal(np.concatenate(parts[name][1]), full[name][1]), name


def test_exported_mask_appends_as_a_boolean_column(ctx):
    t = _table(TILE + 33, 0.05, seed=8)
    _register(ctx, "rm_data", t)
    p, sl = _plan_with_masks(ctx)
    p.execute(ctx, "rm_data")
    by = {name: s for name, s, _ in sl}
    for name in ("terms", "non_negative"):
        m = p.row_mask(by[name])
        vals, valid = _read(m)
        _drop(ctx, f"verdicts_{name}")
        tab = ctx._create(f"verdicts_{name}")
        sc, ar = m.__arrow_c_device_array__()
        # the engine takes a RecordBatch: wrap the exported array as its only column
        st = _append_struct(tab, sc, ar)
        assert st == 0, F.lib().tg_last_error()
        from tests.test_arrow_device import _bytes
        got_vals, _, got_valid = _bytes(ctx, f"verdicts_{name}", "v")
        assert np.array_equal(R.unpack(got_vals.tobytes(), len(vals)) & valid, vals & valid)
        if m.validity_ptr:
            assert np.array_equal(R.unpack(got_valid.tobytes(), len(vals)), valid)


def _append_struct(tab, sc, ar):
    """wraps an exported Boolean device array as the single column `v` of a struct RecordBatch and appends it"""
    from term_b200.api import _capsule_pointer
    from tests.test_arrow_device import ArrowArray, ArrowDeviceArray
    sp, ap = _capsule_pointer(sc, b"arrow_schema"), _capsule_pointer(ar, b"arrow_device_array")
    child_dev = ArrowDeviceArray.from_address(ap)
    child_schema = (C.c_uint8 * 72).from_address(sp)
    name = C.c_char_p(b"v")
    C.c_void_p.from_address(sp + 8).value = C.cast(name, C.c_void_p).value
    kids = (C.POINTER(ArrowArray) * 1)(C.pointer(child_dev.array))
    noop = C.CFUNCTYPE(None, C.c_void_p)(lambda p: None)
    bufs = (C.c_void_p * 1)(0)
    top = ArrowArray(length=child_dev.array.length, null_count=0, offset=0, n_buffers=1, n_children=1, buffers=bufs,
                     children=kids, release=C.cast(noop, C.c_void_p))
    dev = ArrowDeviceArray(array=top, device_id=child_dev.device_id, device_type=child_dev.device_type, sync_event=None)
    schema_kids = (C.c_void_p * 1)(sp)

    class S(C.Structure):
        _fields_ = [("format", C.c_char_p), ("name", C.c_char_p), ("metadata", C.c_void_p), ("flags", C.c_int64),
                    ("n_children", C.c_int64), ("children", C.c_void_p), ("dictionary", C.c_void_p), ("release", C.c_void_p),
                    ("private_data", C.c_void_p)]
    top_schema = S(format=b"+s", name=b"", flags=0, n_children=1, children=C.cast(schema_kids, C.c_void_p), release=C.cast(noop, C.c_void_p))
    st = F.lib().tg_table_append_arrow_device(tab, C.addressof(top_schema), C.addressof(dev))
    _append_struct.keep = (name, kids, noop, bufs, top, dev, schema_kids, top_schema, child_schema)
    return st


def test_full_size_against_torch(ctx):
    import torch
    n = 100_000_000
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(n, device="cuda", generator=g, dtype=torch.float64) * 10
    y = torch.randint(-1000, 1000, (n,), device="cuda", generator=g, dtype=torch.int64)
    t = pa.table({"x": pa.array(x.cpu().numpy()), "y": pa.array(y.cpu().numpy())})
    _register(ctx, "rm_data", t)
    del t
    preds = ["x > 0", "y < 10", "x > -5 AND x < 5", "y >= 0 OR x > 3", "x * 2.0 > y", "y % 7 = 3", "ABS(x) < 1.0", "y + 1 > 500"]
    want = [x > 0, y < 10, (x > -5) & (x < 5), (y >= 0) | (x > 3), x * 2.0 > y.double(), torch.fmod(y, 7) == 3,
            x.abs() < 1.0, y + 1 > 500]
    p = T.api.Plan()
    slots = [F.lib().tg_plan_add_custom_sql(p.handle, e.encode(), None) for e in preds]
    for s in slots:
        p.request_row_mask(s)
    p.execute(ctx, "rm_data")
    from term_b200.distributed import _tensor_from_ptr
    shifts = torch.arange(8, device="cuda", dtype=torch.uint8)
    for e, s, w in zip(preds, slots, want):
        m = p.row_mask(s)
        raw = _tensor_from_ptr(m.values_ptr, (n + 7) // 8, torch.device("cuda", 0), "|u1")[: (n + 7) // 8]
        bits = ((raw.unsqueeze(1) >> shifts) & 1).reshape(-1)[:n].bool()
        assert torch.equal(bits, w), e
        assert p.result(s).metric == float(int(w.sum())) / n
