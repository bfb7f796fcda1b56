"""Key-level row verdicts without a GPU: the reference verdicts reproduce the popcount identities tg_plan_export_key_rows
states on every golden vector of the uniqueness and foreign-key kinds, and tg_plan_request_key_rows /
tg_plan_export_key_rows refuse what they must on a host-only plan."""
import ctypes as C

import pytest

import term_b200 as T
from oracle import term_oracle as O
from term_b200 import _ffi as F
from tests import helpers as H
from tests.key_rows_reference import orphan_rows, popcount, uniqueness_rows

DUP, FIRST, ORPHAN = F.TG_KEY_ROWS_DUPLICATE, F.TG_KEY_ROWS_FIRST, F.TG_KEY_ROWS_ORPHAN
INVALID = 1  # TG_ERR_INVALID_ARG


def _uniqueness_identities(table, columns):
    dup, first, valid = uniqueness_rows(table, columns)
    d = O.distinct_counts(table, columns)
    single = len(columns) == 1
    assert popcount(first, valid) == (d["distinct_nonnull"] if single else d["distinct_all"])
    # singleton groups of non-NULL keys (the oracle's count includes the NULL group of a single column)
    singles = d["singletons"] - (1 if single and d["any_null_rows"] == 1 else 0)
    assert popcount(dup, valid) == sum(valid) - singles
    assert sum(valid) == d["rows"] - (d["any_null_rows"] if single else 0)


def _fk_identities(tables, child, parent, allow_nulls):
    orphan, valid = orphan_rows(tables, child, parent)
    _, total, _ = O.foreign_key(tables, child, parent, allow_nulls)
    nulls = len(valid) - sum(valid)
    assert popcount(orphan, valid) == total - (0 if allow_nulls else nulls)


def test_reference_identities_on_golden_vectors():
    seen = {"uniqueness": 0, "foreign_key": 0}
    for case in H.load_golden():
        op = case["op"]
        if op["kind"] == "uniqueness":
            _uniqueness_identities(H.case_tables(case)["data"], op["columns"])
        elif op["kind"] == "foreign_key":
            tables = H.case_tables(case)
            for allow in (False, True):
                _fk_identities(tables, op["child"], op["parent"], allow)
        else:
            continue
        seen[op["kind"]] += 1
    assert seen["uniqueness"] >= 10 and seen["foreign_key"] >= 5, seen


def test_reference_key_equality():
    import pyarrow as pa
    t = pa.table({"f": pa.array([0.0, -0.0, float("nan"), float("nan"), None, 1.5, None]),
                  "s": pa.array(["a", None, "a", None, "b", "a", None])})
    dup, first, valid = uniqueness_rows(t, ["f"])
    assert valid == [True, True, True, True, False, True, False]
    assert dup == [True, True, True, True, False, False, False]
    assert first == [True, False, True, False, False, True, False]
    dup, first, valid = uniqueness_rows(t, ["f", "s"])  # every tuple differs, NULL components included
    assert all(valid) and not any(dup) and all(first)
    t2 = pa.table({"a": pa.array([None, None, 1], type=pa.int64()), "b": pa.array([None, None, 1], type=pa.int64())})
    dup, first, valid = uniqueness_rows(t2, ["a", "b"])  # (NULL, NULL) twice: a repeated value
    assert all(valid) and dup == [True, True, False] and first == [True, False, True]


def _plan():
    p = T.api.Plan()
    lib = F.lib()
    strs = lambda *a: (C.c_char_p * len(a))(*[s.encode() for s in a])
    A = F.tg_assertion(0, 0.0, 0.0)
    slots = {"uniq_" + str(k): lib.tg_plan_add_uniqueness(p.handle, strs("a"), 1, k, 1.0, A, 0) for k in range(6)}
    slots.update({
        "uniq2": lib.tg_plan_add_uniqueness(p.handle, strs("a", "b"), 2, 5, 1.0, A, 0),
        "fk": lib.tg_plan_add_foreign_key(p.handle, b"data.a", b"ref.a", 0, 10),
        "completeness": lib.tg_plan_add_completeness(p.handle, strs("a"), 1, 1.0, 0, 0),
        "sql": lib.tg_plan_add_custom_sql(p.handle, b"a > 1", None),
        "stat": lib.tg_plan_add_statistic(p.handle, b"a", 0, 0.0, A),
        "acd": lib.tg_plan_add_approx_count_distinct(p.handle, b"a", A),
        "an_distinctness": lib.tg_plan_add_analyzer(p.handle, 5, b"a", None, None),
    })
    assert all(v >= 0 for v in slots.values()), slots
    return p, slots


def test_request_refusals(built_lib):
    p, slots = _plan()
    lib = F.lib()
    for name, s in slots.items():
        for kind in (DUP, FIRST, ORPHAN):
            st = lib.tg_plan_request_key_rows(p.handle, s, kind)
            if name.startswith("uniq"):
                assert st == (0 if kind != ORPHAN else INVALID), (name, kind)
            elif name == "fk":
                assert st == (0 if kind == ORPHAN else INVALID), (name, kind)
            else:
                assert st == F.TG_ERR_UNSUPPORTED, (name, kind)
                assert b"key-level row verdicts are not available" in lib.tg_last_error()
    for kind in (-1, 3, 100):
        assert lib.tg_plan_request_key_rows(p.handle, slots["uniq_0"], kind) == INVALID
        assert lib.tg_plan_request_key_rows(p.handle, slots["fk"], kind) == INVALID
    for bad in (-1, len(slots), 10_000):
        assert lib.tg_plan_request_key_rows(p.handle, bad, DUP) == INVALID
    assert lib.tg_plan_request_key_rows(None, 0, DUP) == INVALID
    # the row-mask entry point still refuses these slots
    assert lib.tg_plan_request_row_mask(p.handle, slots["uniq_0"]) == F.TG_ERR_UNSUPPORTED
    assert lib.tg_plan_request_row_mask(p.handle, slots["fk"]) == F.TG_ERR_UNSUPPORTED


def test_export_refusals(built_lib):
    p, slots = _plan()
    p.request_key_rows(slots["uniq_0"], DUP)
    p.request_key_rows(slots["fk"], ORPHAN)
    cases = [
        (slots["uniq_0"], DUP, INVALID),     # requested, not executed
        (slots["uniq_0"], FIRST, INVALID),   # not requested
        (slots["uniq_1"], DUP, INVALID),     # not requested
        (slots["fk"], ORPHAN, INVALID),      # requested, not executed
        (slots["fk"], DUP, INVALID),         # wrong kind
        (slots["uniq_0"], ORPHAN, INVALID),  # wrong kind
        (slots["sql"], DUP, F.TG_ERR_UNSUPPORTED),        # wrong slot kind
        (-1, DUP, INVALID),
        (999, DUP, INVALID),
    ]
    for s, kind, code in cases:
        with pytest.raises(T.TermGpuError) as e:
            p.key_rows(s, kind)
        assert e.value.code == code, (s, kind)
    sc, ar = (C.c_uint8 * 72)(), (C.c_uint8 * 128)()
    assert F.lib().tg_plan_export_key_rows(p.handle, slots["uniq_0"], DUP, None, ar) == INVALID
    assert F.lib().tg_plan_export_key_rows(p.handle, slots["uniq_0"], DUP, sc, None) == INVALID
    assert F.lib().tg_plan_export_key_rows(None, 0, DUP, sc, ar) == INVALID
