"""Row verdicts without a GPU: the reference masks reproduce the oracle's metric for every golden vector of a row-level
kind, and tg_plan_request_row_mask / tg_plan_export_row_mask refuse what they must on a host-only plan."""
import ctypes as C

import pytest

import term_b200 as T
from term_b200 import _ffi as F
from tests import helpers as H
from tests.row_mask_reference import case_mask, ratio

ROW_KINDS = {"completeness", "custom_sql", "containment", "non_negative", "format", "data_type", "length"}


def test_reference_masks_reproduce_the_oracle_metric():
    seen = 0
    for case in H.load_golden():
        if case["op"]["kind"] not in ROW_KINDS:
            continue
        try:
            mask = case_mask(case)
        except Exception:  # a case whose evaluation fails (missing column, division by zero) has no verdicts
            continue
        if mask is None:
            continue
        want = H.oracle_eval(case)
        got = ratio(mask)
        if case["op"]["kind"] == "completeness" and want.metric is None:
            assert got is None or len(mask[0]) == 0
            continue
        assert got == want.metric, (case.get("name"), got, want.metric)
        seen += 1
    assert seen >= 50


def _plan():
    p = T.api.Plan()
    lib = F.lib()
    strs = lambda *a: (C.c_char_p * len(a))(*[s.encode() for s in a])
    A = F.tg_assertion(0, 0.0, 0.0)
    slots = {
        "completeness": lib.tg_plan_add_completeness(p.handle, strs("a"), 1, 1.0, 0, 0),
        "completeness2": lib.tg_plan_add_completeness(p.handle, strs("a", "b"), 2, 1.0, 0, 0),
        "sql": lib.tg_plan_add_custom_sql(p.handle, b"a > 1", None),
        "uniq": lib.tg_plan_add_uniqueness(p.handle, strs("a"), 1, 0, 1.0, A, 0),
        "stat": lib.tg_plan_add_statistic(p.handle, b"a", 0, 0.0, A),
        "size": lib.tg_plan_add_size(p.handle, A),
        "fk": lib.tg_plan_add_foreign_key(p.handle, b"data.a", b"ref.a", 0, 10),
        "corr": lib.tg_plan_add_correlation(p.handle, b"a", b"b", 0, A),
        "length": lib.tg_plan_add_length(p.handle, b"s", 0, 2, 0),
        "format": lib.tg_plan_add_format(p.handle, b"s", 1, None, 0, 1.0, None),
        "data_type": lib.tg_plan_add_data_type(p.handle, b"s", 0, 1.0),
        "containment": lib.tg_plan_add_containment(p.handle, b"s", strs("x", "y"), 2),
        "non_negative": lib.tg_plan_add_non_negative(p.handle, b"a"),
        "an_completeness": lib.tg_plan_add_analyzer(p.handle, 1, b"a", None, None),
        "an_compliance": lib.tg_plan_add_analyzer(p.handle, 13, None, None, b"a > 0"),
        "an_mean": lib.tg_plan_add_analyzer(p.handle, 2, b"a", None, None),
        "column_count": lib.tg_plan_add_column_count(p.handle, A),
    }
    assert all(v >= 0 for v in slots.values()), slots
    return p, slots


SUPPORTED = {"completeness", "sql", "length", "format", "data_type", "containment", "non_negative", "an_completeness", "an_compliance"}


def test_request_refusals_on_a_host_only_plan(built_lib):
    p, slots = _plan()
    for name, s in slots.items():
        st = F.lib().tg_plan_request_row_mask(p.handle, s)
        if name in SUPPORTED:
            assert st == 0, (name, F.lib().tg_last_error())
        else:
            assert st == F.TG_ERR_UNSUPPORTED, name
            assert b"row verdicts are not available" in F.lib().tg_last_error()
    for bad in (-1, len(slots), 10_000):
        assert F.lib().tg_plan_request_row_mask(p.handle, bad) == 1
    assert F.lib().tg_plan_request_row_mask(None, 0) == 1


def test_export_before_execute_is_an_error(built_lib):
    p, slots = _plan()
    p.request_row_mask(slots["sql"])
    for s in (slots["sql"], slots["length"], slots["uniq"], -1, 999):
        with pytest.raises(T.TermGpuError) as e:
            p.row_mask(s)
        assert e.value.code == 1
    sc, ar = (C.c_uint8 * 72)(), (C.c_uint8 * 128)()
    assert F.lib().tg_plan_export_row_mask(p.handle, slots["sql"], None, ar) == 1
    assert F.lib().tg_plan_export_row_mask(p.handle, slots["sql"], sc, None) == 1
