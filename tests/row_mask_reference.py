"""Reference row verdicts for tg_plan_export_row_mask: per row (value, valid) built from the oracle's own row evaluation
(`_ev` for predicates, `regex_matches` for patterns, the length rule of `length_constraint`), so that
sum(value and valid) / sum(valid) is the metric the oracle reports for the same constraint."""
import numpy as np

from oracle import term_oracle as O


def _rows(table):
    cols = O.table_cols(table)
    names = list(cols)
    for i in range(O.n_rows(cols)):
        row = {}
        for nm in names:
            c = cols[nm]
            v = c.values[i] if c.valid[i] else None
            row[nm] = v.item() if hasattr(v, "item") else v
        yield row


def completeness_mask(table, column):
    """one column: value = the row is non-null; every row counts"""
    valid = [bool(v) for v in O.table_cols(table)[column].valid]
    return valid, [True] * len(valid)


def predicate_mask(table, expression):
    """custom_sql / satisfies / ComplianceAnalyzer: value = the predicate IS TRUE; every row counts"""
    cols = O.table_cols(table)
    ast = O._annotate(O._P(O._tokenize(expression)).or_(), {nm: c.kind for nm, c in cols.items()},
                      {nm: c.temporal_unit for nm, c in cols.items() if c.temporal_unit})
    vals = [O._ev(ast, row) is True for row in _rows(table)]
    return vals, [True] * len(vals)


def containment_mask(table, column, allowed):
    c = O.table_cols(table)[column]
    allowed = set(str(v) for v in allowed)
    return [bool(ok) and str(v) in allowed for v, ok in zip(c.values, c.valid)], [bool(ok) for ok in c.valid]


def non_negative_mask(table, column):
    c = O.table_cols(table)[column]
    return [bool(ok) and float(v) >= 0 for v, ok in zip(c.values, c.valid)], [bool(ok) for ok in c.valid]


def format_mask(table, column, pattern, case_sensitive=True, trim=False, null_is_valid=True):
    ms = O.regex_matches(O.table_cols(table)[column], pattern, not case_sensitive, trim)
    return [m is True or (m is None and null_is_valid) for m in ms], [True] * len(ms)


def data_type_mask(table, column, dtype):
    ms = O.regex_matches(O.table_cols(table)[column], O.DATA_TYPE_PATTERNS[dtype])
    return [m is True for m in ms], [m is not None for m in ms]


def length_mask(table, column, lo, hi=None):
    """value = NULL, or lo <= LENGTH(c) [<= hi] in characters; every row counts"""
    c = O.table_cols(table)[column]
    vals = [not ok or (len(v) >= lo and (hi is None or len(v) <= hi)) for v, ok in zip(c.values, c.valid)]
    return vals, [True] * len(vals)


LENGTH_RANGE = {"Min": lambda a, b: (a, None), "Max": lambda a, b: (0, a), "Between": lambda a, b: (a, b),
                "Exactly": lambda a, b: (a, a), "NotEmpty": lambda a, b: (1, None)}


def case_mask(case):
    """the reference mask of a golden-vector case of a row-level kind, or None for any other case"""
    from tests.helpers import case_tables
    op = case["op"]
    t = case_tables(case).get("data")
    k = op["kind"]
    if k == "completeness" and len(op["columns"]) == 1:
        return completeness_mask(t, op["columns"][0])
    if k == "custom_sql":
        return predicate_mask(t, op["expression"])
    if k == "containment":
        return containment_mask(t, op["column"], op["allowed"])
    if k == "non_negative":
        return non_negative_mask(t, op["column"])
    if k == "format":
        return format_mask(t, op["column"], O.format_pattern(op["format"], op.get("arg"), op.get("flag", False)),
                           op.get("case_sensitive", True), op.get("trim", False), op.get("null_is_valid", True))
    if k == "data_type":
        return data_type_mask(t, op["column"], op["data_type"])
    if k == "length":
        a = op["assertion"]
        return length_mask(t, op["column"], *LENGTH_RANGE[a[0]](*(list(a[1:]) + [0, 0])[:2]))
    return None


def ratio(mask):
    vals, valid = mask
    num = sum(1 for v, ok in zip(vals, valid) if v and ok)
    den = sum(1 for ok in valid if ok)
    return float(num) / float(den) if den else None


def unpack(ptr_bytes, n):
    """LSB-first bitmap bytes -> n booleans"""
    return np.unpackbits(np.frombuffer(ptr_bytes, dtype=np.uint8), bitorder="little")[:n].astype(bool)
