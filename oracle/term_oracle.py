"""CPU oracle — TEST INFRASTRUCTURE ONLY (never imported by term_b200/, never a fallback).

A plain numpy / pure-Python restatement of what the reference (withterm/term, `term-guard` 0.0.2)
computes on the hot path by lowering each constraint / analyzer to a DataFusion SQL aggregate.
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import it.

The arithmetic itself lives in third-party crates that are NOT vendored under /root/reference
(datafusion 50.3.0, arrow 56.2.0, regex 1.12.2 / regex-syntax 0.8.8 — Cargo.lock); this file restates
the published SQL semantics those queries have (SURVEY.md §8c) and the in-tree Rust that follows each
query. Every function cites the reference file:line it follows (paths under term-guard/src/).

PINNING: the reference cannot be built here (no cargo/rustc), so the oracle is pinned against the
reference's own known-answer tests, ported to tests/golden/reference_vectors.json with their file:line
(tests/test_oracle_golden.py). Values no reference test fixes are "parity unpinned" (SURVEY.md §8c last
row): APPROX_PERCENTILE_CONT, CORR with zero variance / n<2, float MIN/MAX with NaN, FK example choice.
"""
import math
import re
from dataclasses import dataclass

try:  # the `regex` module implements UTS#18 \w (Alphabetic + M + Nd + Pc + Join_Control) and simple case
    import regex as _rx  # folding exactly like the Rust regex crate; stdlib `re` differs on combining marks
except Exception:  # pragma: no cover
    _rx = re
from decimal import Decimal
from typing import Dict, List, Optional, Sequence

import numpy as np

SUCCESS, FAILURE, SKIPPED = "success", "failure", "skipped"


@dataclass
class Result:  # core/constraint.rs:40-48
    status: str
    metric: Optional[float] = None
    message: Optional[str] = None


# ------------------------------------------------------------------ Rust formatting ----
def rust_f64(v: float) -> str:
    """`{}` of an f64: shortest round-trip digits, never scientific, integral values without '.0'."""
    if math.isnan(v):
        return "NaN"
    if math.isinf(v):
        return "inf" if v > 0 else "-inf"
    s = format(Decimal(repr(float(v))), "f")
    if "." in s:
        s = s.rstrip("0").rstrip(".")
    if s in ("-0", ""):
        s = "-0" if s == "-0" else "0"
    return s


def rust_prec(v: float, n: int) -> str:
    return format(v, f".{n}f")


# ------------------------------------------------------------------ Assertion / LogicalOperator ----
def assertion_eval(a, value: float) -> bool:
    """constraints/assertion.rs:48-61; a = (kind, x[, y])"""
    k = a[0]
    eps = 1e-10
    if k == "Equals":
        return abs(value - a[1]) < eps
    if k == "NotEquals":
        return abs(value - a[1]) >= eps
    if k == "GreaterThan":
        return value > a[1]
    if k == "GreaterThanOrEqual":
        return value >= a[1]
    if k == "LessThan":
        return value < a[1]
    if k == "LessThanOrEqual":
        return value <= a[1]
    if k == "Between":
        return a[1] <= value <= a[2]
    if k == "NotBetween":
        return value < a[1] or value > a[2]
    raise ValueError(k)


def assertion_desc(a) -> str:
    """constraints/assertion.rs:64-75"""
    k = a[0]
    names = {"Equals": "equals", "NotEquals": "not equals", "GreaterThan": "greater than",
             "GreaterThanOrEqual": "greater than or equal to", "LessThan": "less than",
             "LessThanOrEqual": "less than or equal to"}
    if k in names:
        return f"{names[k]} {rust_f64(a[1])}"
    if k == "Between":
        return f"between {rust_f64(a[1])} and {rust_f64(a[2])}"
    return f"not between {rust_f64(a[1])} and {rust_f64(a[2])}"


def logical_eval(op, results: Sequence[bool]) -> bool:
    """core/logical.rs:69-89; op = ("All",) | ("Any",) | ("Exactly", n) | ("AtLeast", n) | ("AtMost", n)"""
    k = op[0]
    if len(results) == 0:
        return {"All": True, "Any": False, "AtMost": True}.get(k, (op[1] if len(op) > 1 else 0) == 0)
    t = sum(1 for r in results if r)
    if k == "All":
        return t == len(results)
    if k == "Any":
        return t > 0
    if k == "Exactly":
        return t == op[1]
    if k == "AtLeast":
        return t >= op[1]
    if k == "AtMost":
        return t <= op[1]
    raise ValueError(k)


def logical_desc(op) -> str:
    k = op[0]
    return {"All": "all", "Any": "any"}.get(k) or {"Exactly": "exactly", "AtLeast": "at least", "AtMost": "at most"}[k] + f" {op[1]}"


# ------------------------------------------------------------------ column access ----
class Col:
    """values: numpy array (numeric) or list of str; valid: bool mask; kind: 'i64' | 'f64' | 'str' | 'bool'"""

    def __init__(self, values, valid, kind, narrow=None, unsigned=False):
        self.values, self.valid, self.kind = values, np.asarray(valid, dtype=bool), kind
        self.unsigned = unsigned  # SUM of an unsigned column is UInt64: the reference's downcasts fail on it as well
        self.temporal_unit = None  # 'D' (Date32 days) / 's' / 'm' / 'u' / 'n': string literals compared with the column are cast to it
        # Arrow name of a 4-byte numeric source type ("Int32" / "Float32"): DataFusion's MIN / MAX keep that type and the
        # reference's Int64 / Float64 downcasts fail (constraints/statistics.rs:278-308, analyzers/basic/min_max.rs:112-131)
        self.narrow = narrow

    def __len__(self):
        return len(self.valid)


def col_from_arrow(arr) -> Col:
    import pyarrow as pa
    if isinstance(arr, pa.ChunkedArray):
        arr = arr.combine_chunks()
    valid = np.asarray(arr.is_valid())
    t = arr.type
    if pa.types.is_temporal(t):  # dates / times / timestamps / durations: their integer representation (comparisons only)
        ints = arr.cast(pa.int32() if t.bit_width == 32 else pa.int64())
        c = Col(np.asarray(ints.fill_null(0)).astype(np.int64), valid, "i64", str(t))
        if pa.types.is_date32(t):
            c.temporal_unit = "D"
        elif pa.types.is_date64(t):
            c.temporal_unit = "m"
        elif pa.types.is_timestamp(t):
            c.temporal_unit = {"s": "s", "ms": "m", "us": "u", "ns": "n"}[t.unit]
        return c
    if pa.types.is_integer(t):
        vals = np.asarray(arr.fill_null(0)).astype(np.int64)
        names = {pa.int8(): "Int8", pa.int16(): "Int16", pa.int32(): "Int32", pa.uint8(): "UInt8", pa.uint16(): "UInt16", pa.uint32(): "UInt32",
                 pa.uint64(): "UInt64"}
        return Col(vals, valid, "i64", names.get(t), pa.types.is_unsigned_integer(t))
    if pa.types.is_floating(t):
        vals = np.asarray(arr.fill_null(0.0)).astype(np.float64)
        return Col(vals, valid, "f64", "Float32" if pa.types.is_float32(t) else None)
    if pa.types.is_boolean(t):
        return Col(np.asarray(arr.fill_null(False)), valid, "bool")
    return Col(arr.to_pylist(), valid, "str")


def table_cols(table) -> Dict[str, Col]:
    """table: pyarrow.Table / RecordBatch or dict name -> Col"""
    if isinstance(table, dict):
        return table
    return {n: col_from_arrow(table.column(n)) for n in table.schema.names}


def n_rows(cols: Dict[str, Col]) -> int:
    return len(next(iter(cols.values()))) if cols else 0


# ------------------------------------------------------------------ constraints ----
def completeness_column(col: Col, name: str, threshold: float) -> Result:
    """constraints/completeness.rs:137-246: SELECT COUNT(*), COUNT(c)"""
    total = float(len(col))
    if total == 0.0:
        return Result(SKIPPED, None, "No data to validate")
    c = float(int(col.valid.sum())) / total
    if c >= threshold:
        return Result(SUCCESS, c)
    return Result(FAILURE, c, f"Column '{name}' completeness {rust_prec(c * 100.0, 2)}% is below threshold {rust_prec(threshold * 100.0, 2)}%")


def completeness(table, columns, threshold=1.0, op=("All",)) -> Result:
    """core/unified.rs:41-123"""
    cols = table_cols(table)
    columns = [columns] if isinstance(columns, str) else list(columns)
    if len(columns) == 0:
        return Result(SKIPPED, None, "No columns specified")
    rs = [completeness_column(cols[c], c, threshold) for c in columns]
    if len(rs) == 1:
        return rs[0]
    bools = [r.status == SUCCESS for r in rs]
    metrics = [r.metric for r in rs if r.metric is not None]
    metric = sum(metrics) / len(metrics) if metrics else None
    ok = logical_eval(op, bools)
    if ok:
        if op[0] == "All":
            msg = f"All {len(columns)} columns satisfy the constraint"
        elif op[0] == "Any":
            msg = "Columns " + ", ".join(c for c, b in zip(columns, bools) if b) + " satisfy the constraint"
        else:
            msg = None
        return Result(SUCCESS, metric, msg)
    failed = ", ".join(c for c, b in zip(columns, bools) if not b)
    return Result(FAILURE, metric, f"Constraint failed for columns: {failed}. Required: {logical_desc(op)}")


def size(table, assertion) -> Result:
    """constraints/size.rs:53-119: SELECT COUNT(*)"""
    n = float(n_rows(table_cols(table)))
    if assertion_eval(assertion, n):
        return Result(SUCCESS, n)
    return Result(FAILURE, n, f"Size {rust_f64(n)} does not {assertion_desc(assertion)}")


STAT_NAMES = {"Min": "minimum", "Max": "maximum", "Mean": "mean", "Sum": "sum",
              "StandardDeviation": "standard deviation", "Variance": "variance", "Median": "median"}


def wrap_i64(x: int) -> int:
    x &= (1 << 64) - 1
    return x - (1 << 64) if x >= (1 << 63) else x


def stat_value(col: Col, stat: str) -> Optional[float]:
    """MIN|MAX|AVG|SUM|STDDEV|VARIANCE with DataFusion typing (constraints/statistics.rs:45-56,278-308):
    on Int64 columns MIN/MAX/SUM are Int64 (SUM wraps) then cast to f64; AVG/STDDEV/VARIANCE are Float64;
    STDDEV/VARIANCE are the SAMPLE statistics (tests/property_tests.rs:784-793) and NULL for n < 2."""
    v = col.values[col.valid]
    n = len(v)
    if stat in ("Min", "Max", "Sum", "Mean") and n == 0:
        return None
    if stat == "Min":
        return float(v.min())
    if stat == "Max":
        return float(v.max())
    if stat == "Sum":
        if col.kind == "i64":
            return float(wrap_i64(sum(int(x) for x in v)))
        return math.fsum(float(x) for x in v)
    if stat == "Mean":
        return math.fsum(float(x) for x in v) / n
    if stat in ("StandardDeviation", "Variance"):
        if n < 2:
            return None
        f = [float(x) for x in v]
        if not all(math.isfinite(x) for x in f):  # NaN, or inf - inf (math.fsum raises on +inf with -inf): NaN, as DataFusion
            return math.nan
        mean = math.fsum(f) / n
        var = math.fsum((x - mean) ** 2 for x in f) / (n - 1)
        return math.sqrt(var) if stat == "StandardDeviation" else var
    raise ValueError(stat)


def statistic(table, column, stat, assertion) -> Result:
    """constraints/statistics.rs:254-322"""
    col = table_cols(table)[column]
    if (col.narrow and stat in ("Min", "Max")) or (col.unsigned and stat == "Sum"):  # the result array is neither Int64 nor Float64: `Err(TermError::Internal(..))` (:303-307)
        return Result(FAILURE, None, "Error evaluating constraint: Internal error: Failed to extract statistic value")
    v = stat_value(col, stat)
    name = STAT_NAMES[stat]
    if v is None:
        return Result(FAILURE, None, f"{name} is null (no non-null values)")
    if assertion_eval(assertion, v):
        return Result(SUCCESS, v)
    return Result(FAILURE, v, f"{name} {rust_f64(v)} does not {assertion_desc(assertion)}")


def multi_statistic(table, column, stats) -> Result:
    """constraints/statistics.rs:424-504; stats = [(stat, assertion)]"""
    col = table_cols(table)[column]
    failures, metrics = [], []
    for stat, a in stats:
        name = STAT_NAMES[stat]
        if (col.narrow and stat in ("Min", "Max")) or (col.unsigned and stat == "Sum"):  # :481-485
            failures.append(f"Failed to compute {name}")
            continue
        v = stat_value(col, stat)
        if v is None:
            failures.append(f"{name} is null")
            continue
        metrics.append(v)
        if not assertion_eval(a, v):
            failures.append(f"{name} is {rust_f64(v)} which does not {assertion_desc(a)}")
    if not failures:
        return Result(SUCCESS, metrics[0] if metrics else 0.0)
    return Result(FAILURE, None, "; ".join(failures))


# FormatType::get_pattern, constraints/format.rs:217-307 (pattern strings are interface data)
def format_pattern(kind, arg=None, flag=False) -> str:
    if kind == "Regex":
        return arg
    if kind == "Email":
        return r"^[a-zA-Z0-9.!#$%&'*+/=?^_`{|}~-]+@[a-zA-Z0-9](?:[a-zA-Z0-9-]{0,61}[a-zA-Z0-9])?(?:\.[a-zA-Z0-9](?:[a-zA-Z0-9-]{0,61}[a-zA-Z0-9])?)*$"
    if kind == "Url":
        if flag:
            return r"^https?://(?:localhost|(?:[a-zA-Z0-9.-]+\.?[a-zA-Z]{2,}|(?:\d{1,3}\.){3}\d{1,3}))(?::\d+)?(?:/[^\s]*)?$"
        return r"^https?://[a-zA-Z0-9.-]+\.[a-zA-Z]{2,}(?::\d+)?(?:/[^\s]*)?$"
    if kind == "CreditCard":
        return r"^(?:4[0-9]{12}(?:[0-9]{3})?|5[1-5][0-9]{14}|3[47][0-9]{13}|3[0-9]{13}|6(?:011|5[0-9]{2})[0-9]{12})$|^(?:\d{4}[-\s]?){3}\d{4}$"
    if kind == "Phone":
        return {"US": r"^(\+?1[-.\s]?)?\(?([0-9]{3})\)?[-.\s]?([0-9]{3})[-.\s]?([0-9]{4})$",
                "CA": r"^(\+?1[-.\s]?)?\(?([0-9]{3})\)?[-.\s]?([0-9]{3})[-.\s]?([0-9]{4})$",
                "UK": r"^(\+44\s?)?(?:\(?0\d{4}\)?\s?\d{6}|\(?0\d{3}\)?\s?\d{7}|\(?0\d{2}\)?\s?\d{8})$",
                "DE": r"^(\+49\s?)?(?:\(?0\d{2,5}\)?\s?\d{4,12})$",
                "FR": r"^(\+33\s?)?(?:\(?0\d{1}\)?\s?\d{8})$"}.get(arg, r"^[\+]?[1-9][\d]{0,15}$")
    if kind == "PostalCode":
        return {"US": r"^\d{5}(-\d{4})?$", "CA": r"^[A-Za-z]\d[A-Za-z][ -]?\d[A-Za-z]\d$",
                "UK": r"^[A-Z]{1,2}\d[A-Z\d]?\s?\d[A-Z]{2}$", "DE": r"^\d{5}$", "FR": r"^\d{5}$",
                "JP": r"^\d{3}-\d{4}$", "AU": r"^\d{4}$"}.get(arg, r"^[A-Za-z0-9\s-]{3,10}$")
    if kind == "UUID":
        return r"^[0-9a-fA-F]{8}-[0-9a-fA-F]{4}-[1-5][0-9a-fA-F]{3}-[89abAB][0-9a-fA-F]{3}-[0-9a-fA-F]{12}$"
    if kind == "IPv4":
        return r"^(?:(?:25[0-5]|2[0-4][0-9]|[01]?[0-9][0-9]?)\.){3}(?:25[0-5]|2[0-4][0-9]|[01]?[0-9][0-9]?)$"
    if kind == "IPv6":
        return r"^([0-9a-fA-F]{0,4}:){1,7}([0-9a-fA-F]{0,4})?$|^::$|^::1$|^([0-9a-fA-F]{1,4}:)*::([0-9a-fA-F]{1,4}:)*[0-9a-fA-F]{1,4}$"
    if kind == "Json":
        return r"^\s*[\{\[].*[\}\]]\s*$"
    if kind == "Iso8601DateTime":
        return r"^\d{4}-\d{2}-\d{2}T\d{2}:\d{2}:\d{2}(?:\.\d+)?(?:Z|[+-]\d{2}:\d{2})$"
    if kind == "SocialSecurityNumber":
        return r"^(00[1-9]|0[1-9][0-9]|[1-5][0-9]{2}|6[0-5][0-9]|66[0-5]|667|66[89]|6[7-9][0-9]|[7-8][0-9]{2})-?(0[1-9]|[1-9][0-9])-?(000[1-9]|00[1-9][0-9]|0[1-9][0-9]{2}|[1-9][0-9]{3})$"
    raise ValueError(kind)


def format_description(kind, pattern, arg=None, flag=False) -> str:
    """constraints/format.rs:329-361"""
    return {
        "Regex": f"matches pattern '{pattern}'", "Email": "are valid email addresses",
        "Url": "are valid URLs (including localhost)" if flag else "are valid URLs",
        "CreditCard": "contain credit card number patterns" if flag else "are valid credit card numbers",
        "Phone": f"are valid {arg} phone numbers" if arg else "are valid phone numbers",
        "PostalCode": f"are valid {arg} postal codes", "UUID": "are valid UUIDs",
        "IPv4": "are valid IPv4 addresses", "IPv6": "are valid IPv6 addresses",
        "Json": "are valid JSON documents", "Iso8601DateTime": "are valid ISO 8601 date-time strings",
        "SocialSecurityNumber": "contain Social Security Number patterns"}[kind]


def rust_regex_to_python(pattern: str, case_insensitive: bool):
    """Rust `regex` semantics on top of Python `re`: `$` only at the very end (Python's also matches
    before a trailing newline -> rewrite unescaped `$` outside classes to `\\Z`); `\\z` -> `\\Z`;
    `.` already excludes only \\n; Unicode classes by default for str patterns. Inside a multi-line group ((?m), (?ms), ..)
    `$` keeps its multi-line meaning, which is the crate's. Patterns with Unicode properties (\\p), nested classes or class
    set operations are compiled by the `regex` module (V1 syntax = the crate's), which Python's `re` does not parse."""
    import re as _re
    multiline = _re.search(r"\(\?[a-zA-Z]*m[a-zA-Z]*[):]", pattern) is not None and "(?-m" not in pattern
    out, i, in_class = [], 0, False
    while i < len(pattern):
        ch = pattern[i]
        if ch == "\\" and i + 1 < len(pattern):
            nxt = pattern[i + 1]
            if not in_class and nxt == "z":
                out.append(r"\Z")
            elif not in_class and nxt == "A":
                out.append(r"\A")
            else:
                out.append(ch + nxt)
            i += 2
            continue
        if in_class:
            if ch == "]":
                in_class = False
            out.append(ch)
        elif ch == "[":
            in_class = True
            out.append(ch)
            if i + 1 < len(pattern) and pattern[i + 1] == "^":
                out.append("^")
                i += 1
            if i + 1 < len(pattern) and pattern[i + 1] == "]":
                out.append(r"\]")
                i += 1
        elif ch == "$" and not multiline:
            out.append(r"\Z")
        else:
            out.append(ch)
        i += 1
    py = "".join(out)
    if _re.search(r"\\[pP]|&&|--|~~|\[\[(?!:)", pattern):
        import regex as _regex
        return _regex.compile(py, _regex.V1 | (_regex.IGNORECASE if case_insensitive else 0))
    return _rx.compile(py, _rx.IGNORECASE if case_insensitive else 0)


def regex_matches(col: Col, pattern: str, case_insensitive=False, trim=False) -> List[Optional[bool]]:
    """`c ~ 'pat'` / `~*` = Regex::is_match = unanchored search; TRIM strips ASCII space only
    (constraints/format.rs:756-776)"""
    rx = rust_regex_to_python(pattern, case_insensitive)
    out = []
    for s, ok in zip(col.values, col.valid):
        if not ok:
            out.append(None)
            continue
        if trim:
            s = s.strip(" ")
        out.append(rx.search(s) is not None)
    return out


def format_constraint(table, column, kind, threshold, arg=None, flag=False, case_sensitive=True, trim=False,
                      null_is_valid=True) -> Result:
    """constraints/format.rs:740-843"""
    col = table_cols(table)[column]
    pattern = format_pattern(kind, arg, flag)
    ms = regex_matches(col, pattern, not case_sensitive, trim)
    matches = float(sum(1 for m in ms if m is True or (m is None and null_is_valid)))
    total = float(len(ms))
    if total == 0.0:
        return Result(SKIPPED, None, "No data to validate")
    ratio = matches / total
    detect = kind == "CreditCard" and flag
    ok = ratio <= threshold if detect else ratio >= threshold
    if ok:
        return Result(SUCCESS, ratio)
    if detect:
        msg = f"Credit card detection ratio {rust_prec(ratio, 3)} exceeds threshold {rust_prec(threshold, 3)}"
    else:
        msg = (f"Format validation ratio {rust_prec(ratio, 3)} is below threshold {rust_prec(threshold, 3)}"
               f" - values that {format_description(kind, pattern, arg, flag)}")
    return Result(FAILURE, ratio, msg)


def _keys(cols: Dict[str, Col], columns):
    """row keys with None for NULL components"""
    cs = [cols[c] for c in columns]
    n = len(cs[0]) if cs else 0
    out = []
    for i in range(n):
        out.append(tuple((c.values[i].item() if hasattr(c.values[i], "item") else c.values[i]) if c.valid[i] else None for c in cs))
    return out


def distinct_counts(table, columns):
    """The five counts every uniqueness flavour needs (constraints/uniqueness.rs:549-718)."""
    cols = table_cols(table)
    keys = _keys(cols, columns)
    from collections import Counter
    cnt = Counter(keys)
    return dict(
        rows=len(keys),
        distinct_nonnull=sum(1 for k in cnt if all(x is not None for x in k)),
        distinct_all=len(cnt),
        singletons=sum(1 for k, v in cnt.items() if v == 1),
        any_null_rows=sum(1 for k in keys if any(x is None for x in k)),
    )


UNIQ_NAMES = {"FullUniqueness": "full_uniqueness", "Distinctness": "distinctness",
              "UniqueValueRatio": "unique_value_ratio", "PrimaryKey": "primary_key",
              "UniqueWithNulls": "unique_with_nulls", "UniqueComposite": "unique_composite"}


def uniqueness(table, columns, kind, threshold=1.0, assertion=None, null_handling="Exclude") -> Result:
    """constraints/uniqueness.rs:449-482 + SQL generators :549-718 + evaluators :721-852.
    COUNT(DISTINCT c) ignores NULL; COUNT(DISTINCT (a, b)) counts struct values (never NULL);
    multi-column distinctness concatenates COALESCE(..,'<NULL>'); GROUP BY keeps a NULL group."""
    columns = [columns] if isinstance(columns, str) else list(columns)
    d = distinct_counts(table, columns)
    multi = len(columns) > 1
    total = float(d["rows"])
    cde = d["distinct_all"] if multi else d["distinct_nonnull"]
    cols_s = ", ".join(columns)
    if kind in ("FullUniqueness", "UniqueWithNulls", "UniqueComposite"):
        unique = cde
        if kind == "UniqueWithNulls" and not multi:
            if null_handling == "Include":
                unique = d["distinct_all"]
            elif null_handling == "Distinct":
                unique = d["distinct_nonnull"] + d["any_null_rows"]
        if total == 0.0:
            return Result(SKIPPED, None, "No data to validate")
        ratio = float(unique) / total
        if ratio >= threshold:
            return Result(SUCCESS, ratio)
        return Result(FAILURE, ratio, f"Uniqueness ratio {rust_prec(ratio, 3)} is below threshold {rust_prec(threshold, 3)} for columns: {cols_s}")
    if kind in ("Distinctness", "UniqueValueRatio"):
        count = float((d["distinct_all"] if multi else d["distinct_nonnull"]) if kind == "Distinctness" else d["singletons"])
        if total == 0.0:
            return Result(SKIPPED, None, "No data to validate")
        ratio = count / total
        if assertion_eval(assertion, ratio):
            return Result(SUCCESS, ratio)
        return Result(FAILURE, ratio, f"{UNIQ_NAMES[kind]} ratio {rust_prec(ratio, 3)} does not satisfy {assertion_desc(assertion)} for columns: {cols_s}")
    if total == 0.0:
        return Result(SKIPPED, None, "No data to validate")
    nulls = float(d["any_null_rows"])
    if nulls > 0.0:
        return Result(FAILURE, nulls / total, f"Primary key columns contain {rust_f64(nulls)} NULL values: {cols_s}")
    if float(cde) != total:
        return Result(FAILURE, (total - cde) / total, f"Primary key columns contain {rust_f64(total - cde)} duplicate values: {cols_s}")
    return Result(SUCCESS, 1.0)


def pair_values(table, c1, c2):
    cols = table_cols(table)
    a, b = cols[c1], cols[c2]
    m = a.valid & b.valid
    return np.asarray(a.values, dtype=np.float64)[m], np.asarray(b.values, dtype=np.float64)[m]


def pearson(x, y) -> Optional[float]:
    """CORR(x, y): population-moment Pearson over pairwise-complete rows; NULL for n < 2 or zero variance
    (parity unpinned there; the constraint reads NULL as 0.0, constraints/correlation.rs:355-362)."""
    n = len(x)
    if n < 2:
        return None
    mx, my = math.fsum(x) / n, math.fsum(y) / n
    sxy = math.fsum((a - mx) * (b - my) for a, b in zip(x, y))
    sxx = math.fsum((a - mx) ** 2 for a in x)
    syy = math.fsum((b - my) ** 2 for b in y)
    den = math.sqrt(sxx * syy)
    if not den > 0.0:
        return None
    return sxy / den


def covar_samp(x, y) -> Optional[float]:
    n = len(x)
    if n < 2:
        return None
    mx, my = math.fsum(x) / n, math.fsum(y) / n
    return math.fsum((a - mx) * (b - my) for a, b in zip(x, y)) / (n - 1)


def correlation(table, c1, c2, kind, assertion) -> Result:
    """constraints/correlation.rs:299-440"""
    if kind in ("Spearman", "KendallTau", "MutualInformation"):
        return Result(SKIPPED, None, "Correlation type not yet implemented")
    x, y = pair_values(table, c1, c2)
    if kind == "Independence":
        v = abs(pearson(x, y) or 0.0)
        if v <= assertion[1]:
            return Result(SUCCESS, v)
        return Result(FAILURE, v, f"Columns {c1} and {c2} have correlation {rust_f64(v)} exceeding independence threshold {rust_f64(assertion[1])}")
    cov = kind == "Covariance"
    v = (covar_samp(x, y) if cov else pearson(x, y)) or 0.0
    if assertion_eval(assertion, v):
        return Result(SUCCESS, v)
    nm = "covariance" if cov else "Pearson correlation"
    return Result(FAILURE, v, f"{nm} between {c1} and {c2} is {rust_f64(v)} which does not {assertion_desc(assertion)}")


# ---- a tiny independent SQL-predicate evaluator (Python objects, None = NULL) for `satisfies` ----
_TOK = re.compile(r"\s*(?:(\d+\.\d*(?:[eE][+-]?\d+)?|\.\d+(?:[eE][+-]?\d+)?|\d+[eE][+-]?\d+)|(\d+)|'((?:[^']|'')*)'|\"((?:[^\"]|\"\")*)\"|([A-Za-z_][A-Za-z0-9_.]*)|(<=|>=|<>|!=|==|[-+*/%<>=(),]))")


def _tokenize(s):
    out, pos = [], 0
    s = s.rstrip()
    while pos < len(s):
        m = _TOK.match(s, pos)
        if not m:
            raise ValueError(f"bad SQL near {s[pos:]!r}")
        pos = m.end()
        if m.group(1) is not None:
            out.append(("f", float(m.group(1))))
        elif m.group(2) is not None:
            out.append(("i", int(m.group(2))))
        elif m.group(3) is not None:
            out.append(("s", m.group(3).replace("''", "'")))
        elif m.group(4) is not None:
            out.append(("c", m.group(4).replace('""', '"')))
        elif m.group(5) is not None:
            w = m.group(5)
            up = w.upper()
            if up in ("AND", "OR", "NOT", "IS", "NULL", "TRUE", "FALSE", "BETWEEN", "IN", "LIKE", "CASE", "WHEN", "THEN", "ELSE", "END", "AS"):
                out.append(("k", up))
            else:
                out.append(("c", w.lower().split(".")[-1]))
        else:
            out.append(("o", m.group(6)))
    out.append(("e", None))
    return out


class _P:
    def __init__(self, toks):
        self.t, self.i = toks, 0

    def peek(self):
        return self.t[self.i]

    def eat(self, kind=None, val=None):
        k, v = self.t[self.i]
        if (kind and k != kind) or (val is not None and v != val):
            raise ValueError(f"unexpected token {k} {v}")
        self.i += 1
        return v

    def is_(self, kind, val=None):
        k, v = self.t[self.i]
        return k == kind and (val is None or v == val)

    def or_(self):
        l = self.and_()
        while self.is_("k", "OR"):
            self.eat()
            l = ("or", l, self.and_())
        return l

    def and_(self):
        l = self.not_()
        while self.is_("k", "AND"):
            self.eat()
            l = ("and", l, self.not_())
        return l

    def not_(self):
        if self.is_("k", "NOT"):
            self.eat()
            return ("not", self.not_())
        return self.cmp()

    def cmp(self):
        l = self.add()
        while True:
            if self.peek()[0] == "o" and self.peek()[1] in ("=", "==", "<>", "!=", "<", "<=", ">", ">="):
                op = self.eat()
                op = {"==": "=", "!=": "<>"}.get(op, op)
                l = ("cmp", op, l, self.add())
            elif self.is_("k", "IS"):
                self.eat()
                neg = False
                if self.is_("k", "NOT"):
                    self.eat()
                    neg = True
                w = self.eat("k")
                l = ("is", w, neg, l)
            elif self.is_("k", "LIKE") or (self.is_("k", "NOT") and self.t[self.i + 1] == ("k", "LIKE")):
                neg = False
                if self.is_("k", "NOT"):
                    self.eat()
                    neg = True
                self.eat("k", "LIKE")
                e = ("like", l, self.add())
                l = ("not", e) if neg else e
            elif self.is_("k", "BETWEEN") or (self.is_("k", "NOT") and self.t[self.i + 1] in (("k", "BETWEEN"), ("k", "IN"))):
                neg = False
                if self.is_("k", "NOT"):
                    self.eat()
                    neg = True
                if self.is_("k", "BETWEEN"):
                    self.eat()
                    lo = self.add()
                    self.eat("k", "AND")
                    hi = self.add()
                    e = ("and", ("cmp", ">=", l, lo), ("cmp", "<=", l, hi))
                else:
                    self.eat("k", "IN")
                    self.eat("o", "(")
                    e = None
                    while True:
                        it = ("cmp", "=", l, self.add())
                        e = it if e is None else ("or", e, it)
                        if self.is_("o", ","):
                            self.eat()
                            continue
                        break
                    self.eat("o", ")")
                l = ("not", e) if neg else e
            elif self.is_("k", "IN"):
                self.eat()
                self.eat("o", "(")
                e = None
                while True:
                    it = ("cmp", "=", l, self.add())
                    e = it if e is None else ("or", e, it)
                    if self.is_("o", ","):
                        self.eat()
                        continue
                    break
                self.eat("o", ")")
                l = e
            else:
                return l

    def add(self):
        l = self.mul()
        while self.peek()[0] == "o" and self.peek()[1] in "+-":
            op = self.eat()
            l = ("ar", op, l, self.mul())
        return l

    def mul(self):
        l = self.unary()
        while self.peek()[0] == "o" and self.peek()[1] in ("*", "/", "%"):
            op = self.eat()
            l = ("ar", op, l, self.unary())
        return l

    def unary(self):
        if self.is_("o", "-"):
            self.eat()
            return ("neg", self.unary())
        if self.is_("o", "+"):
            self.eat()
            return self.unary()
        return self.prim()

    def prim(self):
        k, v = self.peek()
        if k in ("f", "i", "s"):
            self.eat()
            return ("lit", v)
        if k == "k" and v in ("TRUE", "FALSE", "NULL"):
            self.eat()
            return ("lit", {"TRUE": True, "FALSE": False, "NULL": None}[v])
        if k == "o" and v == "(":
            self.eat()
            e = self.or_()
            self.eat("o", ")")
            return e
        if k == "k" and v == "CASE":
            # CASE [operand] WHEN c THEN x .. [ELSE y] END; the simple form compares the operand with each WHEN value
            self.eat()
            operand = None if self.is_("k", "WHEN") else self.or_()
            arms = []
            while self.is_("k", "WHEN"):
                self.eat()
                c = self.or_()
                if operand is not None:
                    c = ("cmp", "=", operand, c)
                self.eat("k", "THEN")
                arms.append((c, self.or_()))
            other = None
            if self.is_("k", "ELSE"):
                self.eat()
                other = self.or_()
            self.eat("k", "END")
            return ("case", arms, other)
        if k == "c" and v in ("date", "timestamp") and self.t[self.i + 1][0] == "s":  # DATE '..' / TIMESTAMP '..'
            self.eat()
            return ("lit", self.eat("s"))
        if k == "c" and v == "interval" and self.t[self.i + 1][0] == "s":  # INTERVAL '1 day' / INTERVAL '1' DAY
            self.eat()
            text = self.eat("s")
            if self.peek()[0] == "c" and self.peek()[1].rstrip("s") in _INTERVAL_UNITS:
                text += " " + self.eat("c")
            return ("interval", text)
        if k == "c" and v in ("current_timestamp", "current_date") and self.t[self.i + 1] != ("o", "("):
            self.eat()
            return ("fn", v.upper(), [])
        if k == "c" and v == "cast" and self.t[self.i + 1] == ("o", "("):
            self.eat()
            self.eat("o", "(")
            e = self.or_()
            self.eat("k", "AS")
            ty = self.eat("c").upper()
            if ty == "DOUBLE" and self.is_("c", "precision"):
                self.eat()
            self.eat("o", ")")
            return ("cast", "f" if ty in ("DOUBLE", "FLOAT", "REAL", "FLOAT8", "FLOAT4") else "i", e)
        if k == "c":
            self.eat()
            if self.is_("o", "("):
                self.eat()
                args = []
                if not self.is_("o", ")"):
                    while True:
                        args.append(self.or_())
                        if self.is_("o", ","):
                            self.eat()
                            continue
                        break
                self.eat("o", ")")
                return ("fn", v.upper(), args)
            return ("col", v)
        raise ValueError(f"unexpected token {k} {v}")


class DivideByZero(Exception):
    pass


def _static_type(e, kinds):
    """'i' | 'f' | 'b' | 's' | None (a NULL literal) — the SQL type of an expression given the columns' kinds: DataFusion
    coerces the arms of CASE / COALESCE to a common type (Int64 with Float64 -> Float64) before evaluating them"""
    k = e[0]
    if k == "lit":
        v = e[1]
        return None if v is None else "b" if isinstance(v, bool) else "i" if isinstance(v, int) else "f" if isinstance(v, float) else "s"
    if k == "col":
        return {"i64": "i", "f64": "f", "bool": "b", "str": "s"}[kinds[e[1]]]
    if k == "neg":
        return _static_type(e[1], kinds)
    if k == "fn":
        if e[1] == "ABS":
            return _static_type(e[2][0], kinds)
        if e[1] == "COALESCE":
            return _unify([_static_type(a, kinds) for a in e[2]])
        return "i"  # the length functions
    if k == "ar":
        a, b = _static_type(e[2], kinds), _static_type(e[3], kinds)
        return None if a is None or b is None else ("f" if "f" in (a, b) else "i")
    if k == "case":
        return _unify([_static_type(x, kinds) for _, x in e[1]] + ([_static_type(e[2], kinds)] if e[2] is not None else []))
    if k == "cast":
        return e[1]
    return "b"


def _unify(types):
    ts = {t for t in types if t is not None}
    if not ts:
        return None
    return "f" if ts == {"i", "f"} else next(iter(ts))


def temporal_literal(text: str, unit: str) -> int:
    """DataFusion's cast of a string literal to the type of the date / timestamp column it is compared with: 'YYYY-MM-DD' for
    Date32 (days since the epoch); 'YYYY-MM-DD[( |T)hh:mm[:ss[.f]]][Z|+hh:mm]' for timestamps (naive = UTC), in the column's unit"""
    import datetime as _dt
    if unit == "D":
        d = _dt.date.fromisoformat(text)
        return (d - _dt.date(1970, 1, 1)).days
    m = re.fullmatch(r"(\d{4}-\d{2}-\d{2})(?:[ Tt](\d{2}):(\d{2})(?::(\d{2})(?:\.(\d+))?)?)?([Zz]|[+-]\d{2}:?\d{2})?", text)
    if not m:
        raise ValueError(f"Cannot cast string '{text}'")
    d = _dt.date.fromisoformat(m.group(1))
    if int(m.group(2) or 0) > 23 or int(m.group(3) or 0) > 59 or int(m.group(4) or 0) > 59:
        raise ValueError(f"Cannot cast string '{text}'")
    secs = (d - _dt.date(1970, 1, 1)).days * 86400 + int(m.group(2) or 0) * 3600 + int(m.group(3) or 0) * 60 + int(m.group(4) or 0)
    frac_ns = int((m.group(5) or "0")[:9].ljust(9, "0"))
    tz = m.group(6)
    if tz and tz not in "Zz":
        sign = -1 if tz[0] == "-" else 1
        digits = tz[1:].replace(":", "")
        secs -= sign * (int(digits[:2]) * 3600 + int(digits[2:4]) * 60)
    return {"s": secs, "m": secs * 1000 + frac_ns // 1_000_000, "u": secs * 1_000_000 + frac_ns // 1000, "n": secs * 1_000_000_000 + frac_ns}[unit]


_INTERVAL_UNITS = {"year": None, "month": None, "week": 7 * 86400 * 10**9, "day": 86400 * 10**9, "hour": 3600 * 10**9, "minute": 60 * 10**9,
                   "second": 10**9, "millisecond": 10**6, "microsecond": 10**3, "nanosecond": 1}


def query_now_ns() -> int:
    """now() is the query's start time (DataFusion folds it at planning time); TG_FIXED_NOW_NS pins it for the parity tests"""
    import os as _os
    import time as _time
    return int(_os.environ["TG_FIXED_NOW_NS"]) if "TG_FIXED_NOW_NS" in _os.environ else _time.time_ns()


def interval_literal(text: str):
    """'N unit [N unit ..]' -> (months, nanoseconds of the day-time part as an exact Fraction-free integer)"""
    from fractions import Fraction
    months, nanos = 0, Fraction(0)
    parts = re.findall(r"\s*([+-]?\d+(?:\.\d+)?)\s*([A-Za-z]*)", text)
    if not parts or "".join(a + b for a, b in parts).replace(" ", "") != text.replace(" ", ""):
        raise ValueError(f"bad interval {text!r}")
    for num, unit in parts:
        u = (unit.lower() or "second")
        u = u[:-1] if len(u) > 1 and u.endswith("s") else u
        if u in ("year", "month"):
            months += int(num) * (12 if u == "year" else 1)
        else:
            nanos += Fraction(num) * _INTERVAL_UNITS[u]
    return months, int(round(nanos))


def _add_interval(ns: int, months: int, nanos: int, sign: int) -> int:
    """timestamp (ns since the epoch) +/- interval: calendar months first (day clamped to the month's length), then the rest"""
    import calendar
    import datetime as _dt
    if months:
        day_ns = 86400 * 10**9
        days, tod = divmod(ns, day_ns)
        d = _dt.date(1970, 1, 1) + _dt.timedelta(days=days)
        mm = d.year * 12 + (d.month - 1) + sign * months
        y, m = divmod(mm, 12)
        d = _dt.date(y, m + 1, min(d.day, calendar.monthrange(y, m + 1)[1]))
        ns = (d - _dt.date(1970, 1, 1)).days * day_ns + tod
    return ns + sign * nanos


def _has_temporal_fn(e) -> bool:
    if e[0] == "interval" or (e[0] == "fn" and e[1] in ("NOW", "CURRENT_TIMESTAMP", "CURRENT_DATE", "TODAY")):
        return True
    return e[0] == "ar" and e[1] in "+-" and (_has_temporal_fn(e[2]) or _has_temporal_fn(e[3]))


def temporal_const_ns(e, now_ns: int) -> int:
    """a constant instant: string / DATE / TIMESTAMP literal, now() / current_timestamp / current_date / today(), +/- intervals"""
    if e[0] == "lit" and isinstance(e[1], str):
        return temporal_literal(e[1], "n")
    if e[0] == "fn" and e[1] in ("NOW", "CURRENT_TIMESTAMP") and not e[2]:
        return now_ns
    if e[0] == "fn" and e[1] in ("CURRENT_DATE", "TODAY") and not e[2]:
        return now_ns - now_ns % (86400 * 10**9)
    if e[0] == "ar" and e[1] in "+-":
        if e[3][0] == "interval":
            return _add_interval(temporal_const_ns(e[2], now_ns), *interval_literal(e[3][1]), 1 if e[1] == "+" else -1)
        if e[1] == "+" and e[2][0] == "interval":
            return _add_interval(temporal_const_ns(e[3], now_ns), *interval_literal(e[2][1]), 1)
    raise ValueError("unsupported date / timestamp arithmetic")


_UNIT_NS = {"D": 86400 * 10**9, "s": 10**9, "m": 10**6, "u": 10**3, "n": 1}


def _annotate(e, kinds, temporal=None):
    """CASE / COALESCE nodes get their coerced result type appended; string literals compared with a date / timestamp column
    become that column's integer"""
    temporal = temporal or {}
    if not isinstance(e, tuple):
        return e
    if e[0] == "cmp":
        a, b = e[2], e[3]
        for col, lit, flip in ((a, b, False), (b, a, True)):
            if col[0] == "col" and temporal.get(col[1]) and _has_temporal_fn(lit):
                # both sides as exact nanoseconds (DataFusion coerces the coarser side up): no rounding to the column's unit
                x = ("lit", temporal_const_ns(lit, query_now_ns()))
                scaled = ("tscale", col, _UNIT_NS[temporal[col[1]]])
                return ("cmp", e[1], x, scaled) if flip else ("cmp", e[1], scaled, x)
            if col[0] == "col" and temporal.get(col[1]) and lit[0] == "lit" and isinstance(lit[1], str):
                v = ("lit", temporal_literal(lit[1], temporal[col[1]]))
                return ("cmp", e[1], v, col) if flip else ("cmp", e[1], col, v)
    if e[0] == "case":
        arms = [(_annotate(c, kinds, temporal), _annotate(x, kinds, temporal)) for c, x in e[1]]
        return ("case", arms, _annotate(e[2], kinds, temporal) if e[2] is not None else None, _static_type(e, kinds))
    if e[0] == "fn" and e[1] == "COALESCE":
        return ("fn", "COALESCE", [_annotate(a, kinds, temporal) for a in e[2]], _static_type(e, kinds))
    if e[0] == "fn":
        return ("fn", e[1], [_annotate(a, kinds, temporal) for a in e[2]])
    if e[0] == "lit" or e[0] == "col":
        return e
    return tuple(_annotate(x, kinds, temporal) if isinstance(x, tuple) else x for x in e)


def _coerce(v, ty):
    return float(v) if (ty == "f" and v is not None and not isinstance(v, bool)) else v


def _ev(e, row):
    k = e[0]
    if k == "lit":
        return e[1]
    if k == "col":
        return row[e[1]]
    if k == "neg":
        v = _ev(e[1], row)
        return None if v is None else (wrap_i64(-v) if isinstance(v, int) and not isinstance(v, bool) else -v)
    if k == "fn":
        if e[1] == "ABS":
            v = _ev(e[2][0], row)
            return None if v is None else abs(v)
        if e[1] in ("LENGTH", "CHAR_LENGTH", "CHARACTER_LENGTH", "OCTET_LENGTH"):  # DataFusion: characters / bytes of a Utf8 value
            v = _ev(e[2][0], row)
            return None if v is None else (len(v.encode("utf-8")) if e[1] == "OCTET_LENGTH" else len(v))
        if e[1] == "COALESCE":  # the first non-NULL argument, coerced to the common type
            for a in e[2]:
                v = _ev(a, row)
                if v is not None:
                    return _coerce(v, e[3])
            return None
        raise ValueError(e[1])
    if k == "case":  # the first arm whose condition is TRUE (NULL is not), else ELSE, else NULL
        for c, x in e[1]:
            if _ev(c, row) is True:
                return _coerce(_ev(x, row), e[3])
        return _coerce(_ev(e[2], row), e[3]) if e[2] is not None else None
    if k == "cast":
        v = _ev(e[2], row)
        if v is None:
            return None
        if e[1] == "f":
            return float(v)
        if isinstance(v, float):
            raise ValueError("CAST of a floating point value to an integer")
        return v
    if k == "like":
        # arrow-string `like`: `%` any sequence, `_` exactly one character, backslash takes the next character literally
        v, pat = _ev(e[1], row), _ev(e[2], row)
        if v is None or pat is None:
            return None
        rx, i = [], 0
        while i < len(pat):
            ch = pat[i]
            if ch == "\\" and i + 1 < len(pat):
                i += 1
                rx.append(re.escape(pat[i]))
            elif ch == "%":
                rx.append(".*")
            elif ch == "_":
                rx.append(".")
            else:
                rx.append(re.escape(ch))
            i += 1
        return re.fullmatch("".join(rx), v, re.DOTALL) is not None
    if k == "ar":
        a, b = _ev(e[2], row), _ev(e[3], row)
        if a is None or b is None:
            return None
        ints = isinstance(a, int) and isinstance(b, int)
        if e[1] == "+":
            return wrap_i64(a + b) if ints else float(a) + float(b)
        if e[1] == "-":
            return wrap_i64(a - b) if ints else float(a) - float(b)
        if e[1] == "*":
            return wrap_i64(a * b) if ints else float(a) * float(b)
        if e[1] == "/":
            if ints:
                if b == 0:
                    raise DivideByZero()
                q = abs(a) // abs(b)
                return wrap_i64(q if (a >= 0) == (b >= 0) else -q)
            fb = float(b)
            fa = float(a)
            if fb == 0.0:
                return math.nan if fa == 0.0 or math.isnan(fa) else math.copysign(math.inf, fa) * math.copysign(1.0, fb)
            return fa / fb
        if e[1] == "%":
            if b == 0:
                raise DivideByZero()
            if ints:  # truncated remainder (sign of the dividend), exact beyond 2^53
                r = abs(a) % abs(b)
                return r if a >= 0 else -r
            return int(math.fmod(a, b))
    if k == "tscale":  # a date / timestamp value in nanoseconds (Python integers: exact)
        v = _ev(e[1], row)
        return None if v is None else v * e[2]
    if k == "cmp":
        a, b = _ev(e[2], row), _ev(e[3], row)
        if a is None or b is None:
            return None
        if not (isinstance(a, int) and isinstance(b, int)) and not isinstance(a, str):
            a, b = float(a), float(b)
        return {"=": a == b, "<>": a != b, "<": a < b, "<=": a <= b, ">": a > b, ">=": a >= b}[e[1]]
    if k == "and":
        a, b = _ev(e[1], row), _ev(e[2], row)
        if a is False or b is False:
            return False
        if a is None or b is None:
            return None
        return True
    if k == "or":
        a, b = _ev(e[1], row), _ev(e[2], row)
        if a is True or b is True:
            return True
        if a is None or b is None:
            return None
        return False
    if k == "not":
        a = _ev(e[1], row)
        return None if a is None else (not a)
    if k == "is":
        a = _ev(e[3], row)
        r = {"NULL": a is None, "TRUE": a is True, "FALSE": a is False}[e[1]]
        return (not r) if e[2] else r
    raise ValueError(k)


def predicate_counts(table, expression):
    """COUNT(CASE WHEN expr THEN 1 END), COUNT(*) — rows where expr is NULL are not counted
    (constraints/custom_sql.rs:203-209)"""
    cols = table_cols(table)
    ast = _annotate(_P(_tokenize(expression)).or_(), {nm: c.kind for nm, c in cols.items()},
                    {nm: c.temporal_unit for nm, c in cols.items() if c.temporal_unit})
    n = n_rows(cols)
    names = list(cols)
    sat = 0
    for i in range(n):
        row = {}
        for nm in names:
            c = cols[nm]
            if not c.valid[i]:
                row[nm] = None
            else:
                v = c.values[i]
                row[nm] = v.item() if hasattr(v, "item") else v
        if _ev(ast, row) is True:
            sat += 1
    return sat, n


def custom_sql(table, expression, hint=None) -> Result:
    """constraints/custom_sql.rs:195-282"""
    try:
        sat, total = predicate_counts(table, expression)
    except DivideByZero:
        return Result(FAILURE, None, f"SQL execution error: Arrow error: Divide by zero error. Expression: '{expression}'")
    if total == 0:
        return Result(SKIPPED, None, "No data to validate")
    ratio = float(sat) / float(total)
    if ratio == 1.0:
        return Result(SUCCESS, ratio)
    failed = int(float(total) - float(sat))
    msg = f"{hint} ({failed} rows failed the condition)" if hint is not None else f"Custom SQL condition not satisfied for {failed} rows. Expression: '{expression}'"
    return Result(FAILURE, ratio, msg)


LENGTH_NAMES = {"Min": "min_length", "Max": "max_length", "Between": "length_between", "Exactly": "exact_length", "NotEmpty": "not_empty"}


def length_constraint(table, column, kind, a=0, b=0) -> Result:
    """constraints/length.rs:150-226: COUNT(CASE WHEN <cond on LENGTH(c)> OR c IS NULL THEN 1 END) * 1.0 /
    NULLIF(COUNT(*), 0); LENGTH counts characters (Unicode scalar values); Success iff ratio >= 1.0."""
    c = table_cols(table)[column]
    n = len(c.valid)
    if n == 0:
        return Result(SKIPPED, None, "No data to validate")
    lo, hi, desc = {"Min": (a, None, f"at least {a} characters"), "Max": (0, a, f"at most {a} characters"),
                    "Between": (a, b, f"between {a} and {b} characters"), "Exactly": (a, a, f"exactly {a} characters"),
                    "NotEmpty": (1, None, "not empty")}[kind]
    ok = 0
    for v, valid in zip(c.values, c.valid):
        if not valid:
            ok += 1
            continue
        L = len(v)  # Python str: code points == Unicode scalar values for valid UTF-8
        if L >= lo and (hi is None or L <= hi):
            ok += 1
    ratio = float(ok) * 1.0 / float(n)
    if ratio >= 1.0:
        return Result(SUCCESS, ratio)
    return Result(FAILURE, ratio, f"Length constraint failed: {rust_prec(ratio * 100.0, 2)}% of values are {desc}")


def containment(table, column, allowed) -> Result:
    """constraints/values.rs:232-296: valid = COUNT(CASE WHEN c IN (..) ..), total = COUNT(*) WHERE c IS NOT NULL"""
    c = table_cols(table)[column]
    allowed = set(str(v) for v in allowed)
    vals = [v for v, ok in zip(c.values, c.valid) if ok]
    total = float(len(vals))
    if total == 0.0:
        return Result(SKIPPED, None, "No non-null data to validate")
    valid = float(sum(1 for v in vals if str(v) in allowed))
    ratio = valid / total
    if ratio == 1.0:
        return Result(SUCCESS, ratio)
    return Result(FAILURE, ratio, f"{rust_f64(total - valid)} values are not in the allowed set")


def non_negative(table, column) -> Result:
    """constraints/values.rs:357-414: COUNT(CASE WHEN CAST(c AS DOUBLE) >= 0 ..), COUNT(*) WHERE c IS NOT NULL"""
    c = table_cols(table)[column]
    vals = [float(v) for v, ok in zip(c.values, c.valid) if ok]
    total = float(len(vals))
    if total == 0.0:
        return Result(SKIPPED, None, "No non-null data to validate")
    nn = float(sum(1 for v in vals if v >= 0))  # NaN >= 0 is false here; Arrow's total order puts NaN last (unpinned)
    ratio = nn / total
    if ratio == 1.0:
        return Result(SUCCESS, ratio)
    return Result(FAILURE, ratio, f"{rust_f64(total - nn)} values are negative")


DATA_TYPE_PATTERNS = {"Integer": r"^-?\d+$", "Float": r"^-?\d*\.?\d+([eE][+-]?\d+)?$", "Boolean": r"^(true|false|TRUE|FALSE|True|False|0|1)$",
                      "Date": r"^\d{4}-\d{2}-\d{2}$", "Timestamp": r"^\d{4}-\d{2}-\d{2}[ T]\d{2}:\d{2}:\d{2}", "String": r".*"}


def data_type(table, column, dtype, threshold) -> Result:
    """constraints/values.rs:104-165: matches = COUNT(CASE WHEN c ~ pattern ..), total = COUNT(*) WHERE c IS NOT NULL"""
    ms = [m for m in regex_matches(table_cols(table)[column], DATA_TYPE_PATTERNS[dtype]) if m is not None]
    total = float(len(ms))
    if total == 0.0:
        return Result(SKIPPED, None, "No non-null data to validate")
    matches = float(sum(1 for m in ms if m))
    ratio = matches / total
    if ratio >= threshold:
        return Result(SUCCESS, ratio)
    return Result(FAILURE, ratio, f"Data type conformance {rust_f64(ratio)} is below threshold {rust_f64(threshold)}")


def column_count(table, assertion) -> Result:
    """constraints/column_count.rs:43-85"""
    n = float(len(table_cols(table)))
    if assertion_eval(assertion, n):
        return Result(SUCCESS, n)
    return Result(FAILURE, n, f"Column count {rust_f64(n)} does not satisfy assertion {assertion_desc(assertion)}")


def unified_data_type(table, column, kind, predicate=None, description="", threshold=None, expected=None, actual_type=None) -> Result:
    """constraints/datatype.rs:296-431 (the unified DataTypeConstraint): SpecificType compares the schema's `{:?}`; Consistency is
    the reference's placeholder (0.95); the other validations count `predicate` over the non-NULL rows:
    SELECT COUNT(*), SUM(CASE WHEN pred THEN 1 ELSE 0 END) FROM t WHERE col IS NOT NULL — Success iff every one satisfies it."""
    cols = table_cols(table)
    if column not in cols:
        raise KeyError(column)
    if kind == "specific":
        if actual_type == expected:
            return Result(SUCCESS, 1.0, f"Column '{column}' has expected type {expected}")
        return Result(FAILURE, 0.0, f"Column '{column}' has type {actual_type}, expected {expected}")
    if kind == "consistency":
        ok = 0.95 >= threshold
        return Result(SUCCESS if ok else FAILURE, 0.95, f"Type consistency {95.0:.1f}% {'meets' if ok else 'below'} threshold {threshold * 100.0:.1f}%")
    c = cols[column]
    # (WHERE col IS NOT NULL filters first: a predicate that ignores the column must not count its NULL rows)
    sat_nn, _ = predicate_counts(table, f'"{column}" IS NOT NULL AND ({predicate})')
    total = int(np.count_nonzero(c.valid))
    rate = sat_nn / total if total else float("nan")
    pct = "NaN" if rate != rate else f"{rate * 100.0:.1f}"
    return Result(SUCCESS if rate >= 1.0 else FAILURE, rate, f"{pct}% of values satisfy {description}")


def temporal_ordering(table, kind, args, allow_nulls=False, tolerance_seconds=0) -> Result:
    """constraints/temporal_ordering.rs:336-600 on the raw Arrow arrays (no SQL evaluator): total_rows = rows the WHERE clause
    keeps, violations = those whose comparison is not TRUE (NULL counts as a violation when NULLs are allowed through).
    kind: 'before_after' (before, after, allow_equal) — compares with `>` when allow_equal, `>=` otherwise, as the reference
    does —, 'date_range' (column, min, max), 'business_hours' (column, 'HH:MM', 'HH:MM', weekdays_only); timestamps are naive UTC."""
    import pyarrow as pa
    units = {"s": 10**9, "ms": 10**6, "us": 10**3, "ns": 1}

    def ns_of(name):
        a = table.column(name).combine_chunks()
        u = units[a.type.unit]
        return [None if v is None else v * u for v in a.cast(pa.int64()).to_pylist()]

    day = 86400 * 10**9
    if kind == "before_after":
        b, a, allow_equal = args
        before, after = ns_of(b), ns_of(a)
        rows = [(x, y) for x, y in zip(before, after) if allow_nulls or (x is not None and y is not None)]
        tol = tolerance_seconds * 10**9 if tolerance_seconds > 0 else 0
        good = sum(1 for x, y in rows if x is not None and y is not None and (y > x + tol if allow_equal else y >= x + tol))
        what = f"Temporal ordering violation: {{v}} records where '{b}' is not before '{a}'"
    elif kind == "date_range":
        c, lo, hi = args
        vals = ns_of(c)
        lo_ns = temporal_literal(lo, "n") if lo is not None else None
        hi_ns = temporal_literal(hi, "n") if hi is not None else None
        rows = [v for v in vals if allow_nulls or v is not None]
        good = sum(1 for v in rows if v is not None and (lo_ns is None or v >= lo_ns) and (hi_ns is None or v <= hi_ns))
        what = f"Date range violation: {{v}} records with '{c}' outside valid range"
    else:
        c, start, end, weekdays = args
        vals = ns_of(c)
        sec = lambda hhmm: (int(hhmm[:2]) * 3600 + int(hhmm[3:5]) * 60) * 10**9
        rows = []
        for v in vals:
            if v is None:
                if allow_nulls and not weekdays:  # EXTRACT(DOW FROM NULL) BETWEEN .. is NULL: the WHERE clause drops the row
                    rows.append(v)
                continue
            if weekdays and not 1 <= ((v // day) + 4) % 7 <= 5:   # Sunday = 0; 1970-01-01 was a Thursday
                continue
            rows.append(v)
        good = sum(1 for v in rows if v is not None and sec(start) <= v % day <= sec(end))
        what = f"Business hours violation: {{v}} records with '{c}' outside business hours"
    total, violations = len(rows), len(rows) - good
    if violations == 0:
        return Result(SUCCESS, 1.0)
    rate = (total - violations) / total if total > 0 else 1.0
    return Result(FAILURE, rate, what.format(v=violations) + f" ({rate * 100.0:.2f}% compliance)")


def cross_table_sum(left_table, left_col, right_table, right_col, left_name, right_name, tolerance=0.0, max_violations=100) -> Result:
    """constraints/cross_table_sum.rs:196-215, 560-628 (no grouping): COALESCE(SUM(l), 0.0) vs COALESCE(SUM(r), 0.0); Success with
    the absolute difference as the metric when it is within the tolerance. Sums with math.fsum (exactly rounded)."""
    def total(table, col):
        c = table_cols(table)[col]
        vals = [float(v) for v, ok in zip(c.values, c.valid) if ok]
        return math.fsum(vals) if vals else 0.0
    left, right = total(left_table, left_col), total(right_table, right_col)
    diff = abs(left - right)
    if not diff > tolerance:
        return Result(SUCCESS, diff)
    tol = f" (tolerance: {tolerance:.4f})" if tolerance > 0.0 else " (exact match required)"
    if max_violations > 0:
        ex = f"Group 'ALL': {left_name} = {left:.4f}, {right_name} = {right:.4f} (diff: {diff:.4f})"
        return Result(FAILURE, diff, f"Cross-table sum mismatch: 1/1 overall totals failed validation{tol}. Examples: [{ex}]")
    return Result(FAILURE, diff, f"Cross-table sum mismatch: 1/1 overall totals failed validation{tol}, total sums: {rust_f64(left)} vs {rust_f64(right)} "
                                 f"(max diff: {diff:.4f})")


def join_coverage(left, lk, right, rk, left_name, right_name, expected=1.0, coverage="Left", distinct_only=False, max_examples=100) -> Result:
    """constraints/join_coverage.rs:186-426 with the joins spelled out (any key multiplicities): LEFT JOIN rows = every left row once
    per matching right row (once when there is none); matched = those with a partner. distinct_only divides the matched ROWS by
    COUNT(DISTINCT left key), as the reference's query does. NULL keys never match."""
    from collections import Counter

    def keys(table, col):
        c = table_cols(table)[col]
        return [v if ok else None for v, ok in zip(c.values, c.valid)]

    L, R = keys(left, lk), keys(right, rk)
    cl, cr = Counter(k for k in L if k is not None), Counter(k for k in R if k is not None)

    def one_way(rows, other):  # (join rows, matched join rows) of `rows` OUTER JOIN other
        total = sum(max(other.get(k, 0), 1) if k is not None else 1 for k in rows)
        matched = sum(other.get(k, 0) for k in rows if k is not None)
        return total, matched

    div = lambda a, b: a / b if b else float("nan")
    tl, ml = one_way(L, cr)
    tr, mr = one_way(R, cl)
    if coverage == "Left":
        rate = div(ml, len(cl) if distinct_only else tl)
    elif coverage == "Right":
        rate = div(mr, tr)
    else:
        a, b = div(ml, tl), div(mr, tr)
        rate = float("nan") if (a != a or b != b) else min(a, b)
    if rate >= expected:
        return Result(SUCCESS, rate)
    unmatched = {k for k in L if k is None or k not in cr}
    shown = min(len(unmatched), max_examples)
    ex = f" ({shown} unmatched examples found)" if max_examples > 0 and shown > 0 else ""
    arrow = {"Left": "->", "Right": "<-", "Bidirectional": "<->"}[coverage]
    pct = lambda x: "NaN" if x != x else f"{x * 100.0:.2f}"
    return Result(FAILURE, rate, f"Join coverage constraint failed: {left_name} {arrow} {right_name} coverage is {pct(rate)}% (expected: {pct(expected)}%){ex}")


class OHistogram:
    """constraints/histogram.rs:25-127 — buckets [(value, count, ratio)] ordered by count DESC, value ASC"""

    def __init__(self, buckets, total_count, null_count):
        self.buckets, self.total_count, self.null_count, self.distinct_count = buckets, total_count, null_count, len(buckets)

    def most_common_ratio(self): return self.buckets[0][2] if self.buckets else 0.0
    def least_common_ratio(self): return self.buckets[-1][2] if self.buckets else 0.0
    def bucket_count(self): return len(self.buckets)
    def top_n(self, n): return [(v, r) for v, _, r in self.buckets[:n]]
    def get_value_ratio(self, value): return next((r for v, _, r in self.buckets if v == value), None)
    def null_ratio(self): return 0.0 if self.total_count == 0 else self.null_count / self.total_count
    def follows_power_law(self, top_n, threshold): return sum((r for _, _, r in self.buckets[:top_n]), 0.0) >= threshold

    def is_roughly_uniform(self, threshold):
        if not self.buckets:
            return True
        return False if self.least_common_ratio() == 0.0 else self.most_common_ratio() / self.least_common_ratio() <= threshold

    def entropy(self):
        e = 0.0
        for _, _, r in self.buckets:
            if r > 0.0:
                e += -r * math.log(r)
        return e


def histogram_of(table, column) -> OHistogram:
    """the query of constraints/histogram.rs:214-241: GROUP BY CAST(c AS VARCHAR) over the non-NULL rows, ratio = count * 1.0 /
    (total - nulls), ORDER BY count DESC, value (VARCHAR: byte order). Utf8, integer and Boolean columns."""
    c = table_cols(table)[column]
    counts = {}
    nulls = 0
    for v, ok in zip(c.values, c.valid):
        if not ok:
            nulls += 1
            continue
        if c.kind == "bool":
            k = "true" if v else "false"
        elif c.kind == "str":
            k = v
        elif c.kind == "i64":
            k = str(int(v))
        else:
            raise ValueError("histogram of a floating-point column: CAST AS VARCHAR formatting is not restated")
        counts[k] = counts.get(k, 0) + 1
    total = len(c.values)
    items = sorted(counts.items(), key=lambda kv: (-kv[1], kv[0].encode("utf-8")))
    return OHistogram([(k, n, n * 1.0 / (total - nulls)) for k, n in items], total, nulls)


def histogram_constraint(table, column, assertion, description="custom assertion") -> Result:
    """constraints/histogram.rs:208-413: Skipped without a non-NULL row; metric = entropy; the failure message at :371-381"""
    h = histogram_of(table, column)
    if not h.buckets:
        return Result(SKIPPED, None, "No data to analyze")
    if assertion(h):
        return Result(SUCCESS, h.entropy())
    return Result(FAILURE, h.entropy(), f"Histogram assertion '{description}' failed for column '{column}'. Distribution: {h.distinct_count} distinct values, "
                                        f"most common ratio: {h.most_common_ratio() * 100.0:.2f}%, null ratio: {h.null_ratio() * 100.0:.2f}%")


def an_histogram(table, column, num_buckets):
    """analyzers/advanced/histogram.rs:184-358 -> dict(total_count, min, max, sum, sum_squared, mean, std_dev,
    buckets=[(lower, upper, count)]); Float64 columns only (the reference's downcasts reject Int64)."""
    c = table_cols(table)[column]
    nb = min(max(int(num_buckets), 1), 1000)
    vals = np.asarray(c.values, dtype=np.float64)[c.valid]
    n = len(vals)
    if n == 0:
        return dict(total_count=0, min=0.0, max=0.0, sum=0.0, sum_squared=0.0, mean=0.0, std_dev=0.0, buckets=[])
    mn, mx = float(vals.min()), float(vals.max())
    s, s2 = math.fsum(vals), math.fsum(vals * vals)
    rng = mx - mn
    w = rng / nb if (rng > 0.0 and nb > 1) else 1.0
    lowers = [mn + (i * w) for i in range(nb)]
    uppers = [(mx + w * 0.001) if i == nb - 1 else mn + ((i + 1) * w) for i in range(nb)]
    counts = [0] * nb
    for v in vals:
        b = nb  # ELSE {num_buckets}
        for i in range(nb):
            if v >= lowers[i] and v < uppers[i]:
                b = i + 1
                break
        counts[b - 1] += 1
    mean = s / n
    std = math.sqrt(max(s2 / n - mean * mean, 0.0)) if n > 1 else 0.0
    return dict(total_count=n, min=mn, max=mx, sum=s, sum_squared=s2, mean=mean, std_dev=std, buckets=list(zip(lowers, uppers, counts)))


def approx_count_distinct(table, column, assertion) -> Result:
    """constraints/approx_count_distinct.rs:49-134: SELECT APPROX_DISTINCT(c) (HyperLogLog; the reference's tests only
    assert ranges). This restatement returns the exact distinct count, which every HLL error bound contains."""
    d = float(distinct_counts(table, [column])["distinct_nonnull"])
    if assertion_eval(assertion, d):
        return Result(SUCCESS, d)
    return Result(FAILURE, d, f"Approximate distinct count {rust_f64(d)} does not satisfy assertion {assertion_desc(assertion)} for column '{column}'")


def foreign_key(tables, child, parent, allow_nulls=False, max_examples=100):
    """constraints/foreign_key.rs:307-410: LEFT JOIN child->parent WHERE parent.col IS NULL [AND child.col IS
    NOT NULL] -> COUNT(*), COUNT(DISTINCT child.col). Returns (Result, total, unique)."""
    ct, cc = child.split(".")
    pt, pc = parent.split(".")
    ccol = table_cols(tables[ct])[cc]
    pcol = table_cols(tables[pt])[pc]
    pset = set((v.item() if hasattr(v, "item") else v) for v, ok in zip(pcol.values, pcol.valid) if ok)
    total, uniq = 0, set()
    for v, ok in zip(ccol.values, ccol.valid):
        if not ok:
            if not allow_nulls:
                total += 1
            continue
        v = v.item() if hasattr(v, "item") else v
        if v not in pset:
            total += 1
            uniq.add(v)
    if total == 0:
        return Result(SUCCESS, None, None), 0, 0
    msg = (f"Foreign key constraint violation: {total} values in '{child}' do not exist in '{parent}' "
           f"(total: {total}, unique: {len(uniq)})")  # examples are an unordered DISTINCT..LIMIT: unpinned
    return Result(FAILURE, float(total), msg), total, len(uniq)


# ------------------------------------------------------------------ analyzers ----
def an_completeness(table, column):
    """analyzers/basic/completeness.rs:58-146 -> (total, non_null, metric)"""
    c = table_cols(table)[column]
    t, nn = len(c), int(c.valid.sum())
    return t, nn, (1.0 if t == 0 else nn / t)


def an_distinctness(table, column):
    """analyzers/basic/distinctness.rs:105-153: COUNT(c), COUNT(DISTINCT c)"""
    d = distinct_counts(table, [column])
    nn = d["rows"] - d["any_null_rows"]
    return nn, d["distinct_nonnull"], (1.0 if nn == 0 else d["distinct_nonnull"] / nn)


def an_stddev(table, column):
    """analyzers/advanced/standard_deviation.rs:163-279 (state -> metric map)"""
    c = table_cols(table)[column]
    v = [float(x) for x in c.values[c.valid]]
    n = len(v)
    if n == 0:
        return None
    s, ss = math.fsum(v), math.fsum(x * x for x in v)
    mean = s / n
    m2 = math.fsum((x - mean) ** 2 for x in v)
    out = {"count": float(n), "mean": mean, "std_dev": math.sqrt(m2 / n), "variance": m2 / n}
    if n > 1:
        out["sample_std_dev"] = math.sqrt(m2 / (n - 1))
        out["sample_variance"] = m2 / (n - 1)
    if abs(mean) >= 2.220446049250313e-16:
        out["coefficient_of_variation"] = math.sqrt(m2 / n) / abs(mean)
    return dict(count=n, sum=s, sum_squared=ss, mean=mean, metric=out)


def an_correlation(table, c1, c2, kind="pearson"):
    """analyzers/advanced/correlation.rs:227-435. Spearman = Pearson over RANK() (competition/min ranks)."""
    x, y = pair_values(table, c1, c2)
    if kind == "spearman":
        from scipy.stats import rankdata
        x = rankdata(x, method="min").astype(np.float64)
        y = rankdata(y, method="min").astype(np.float64)
    n = len(x)
    if n < 2:
        return math.nan
    if kind == "covariance":
        return covar_samp(x, y)
    r = pearson(x, y)
    return 0.0 if r is None else r


def grouped_completeness(table, column, group_columns):
    """analyzers/basic/grouped_completeness.rs:131-239: GROUP BY g.. -> {key: (total, non_null)}"""
    cols = table_cols(table)
    tgt = cols[column]
    keys = _keys(cols, group_columns)
    out = {}
    for k, ok in zip(keys, tgt.valid):
        t = out.setdefault(k, [0, 0])
        t[0] += 1
        t[1] += int(ok)
    return out


def exact_quantile(values: np.ndarray, q: float) -> float:
    """the reference's own accuracy harness: sorted[min(floor(n*q), n-1)] (tests/tpc_integration_tests.rs:533-551)"""
    s = np.sort(values)
    return float(s[min(int(len(s) * q), len(s) - 1)])


def rank_error(values_sorted: np.ndarray, estimate: float, q: float) -> float:
    """|rank(estimate)/n - q| with the most favourable rank among ties"""
    n = len(values_sorted)
    lo = np.searchsorted(values_sorted, estimate, side="left") / n
    hi = np.searchsorted(values_sorted, estimate, side="right") / n
    if lo <= q <= hi:
        return 0.0
    return min(abs(lo - q), abs(hi - q))


def kll_exact_quantile(values: np.ndarray, q: float) -> float:
    """KllSketch::get_quantile with every item still at level 0 (weight 1), analyzers/advanced/kll_sketch.rs:246-318:
    phi 0 / 1 => min / max, else the first sorted item whose cumulative weight reaches ceil(phi * n); NaN skipped
    on update (:197-199)"""
    s = np.sort(values[~np.isnan(values)])
    if len(s) == 0:
        return 0.0
    if q <= 0.0:
        return float(s[0])
    if q >= 1.0:
        return float(s[-1])
    target = max(1, math.ceil(q * len(s)))
    return float(s[min(target, len(s)) - 1])


def quantile_constraint(table, column, mode, checks=(), quantiles=(), strict=False, quantile_fn=kll_exact_quantile) -> Result:
    """constraints/quantile.rs:282-482. mode: "Single" [(q, assertion)], "Multiple" [(q, assertion)...],
    "Monotonic" quantiles + strict, anything else => the catch-all Skipped arm (:474-479). The quantile VALUES come
    from quantile_fn (APPROX_PERCENTILE_CONT in the reference — parity unpinned, SURVEY §8c; here the KLL rule);
    a NULL aggregate (no non-null rows) is read as 0.0 (`.value(0)` without a null check, :311-316)."""
    col = table_cols(table)[column]
    vals = np.asarray(col.values, dtype=np.float64)[col.valid]

    def qv(q):
        return quantile_fn(vals, q) if len(vals) else 0.0

    if mode == "Single":
        q, a = checks[0]
        v = qv(q)
        if assertion_eval(a, v):
            return Result(SUCCESS, v)
        return Result(FAILURE, v, f"Quantile {rust_f64(q)} is {rust_f64(v)} which does not {assertion_desc(a)}")
    if mode == "Multiple":
        failures = []
        for q, a in checks:
            v = qv(q)
            if not assertion_eval(a, v):
                failures.append(f"Q{int(q * 100.0)} is {rust_f64(v)} which does not {assertion_desc(a)}")
        return Result(SUCCESS, None) if not failures else Result(FAILURE, None, "; ".join(failures))
    if mode == "Monotonic":
        v = [qv(q) for q in quantiles]
        ok = all((b > a) if strict else (b >= a) for a, b in zip(v, v[1:]))
        if ok:
            return Result(SUCCESS, None)
        dbg = ", ".join(rust_f64(x) if any(c in rust_f64(x) for c in ".eN") or math.isinf(x) else rust_f64(x) + ".0" for x in v)
        return Result(FAILURE, None, f"Quantiles are not {'strictly' if strict else ''} monotonic: [{dbg}]")
    return Result(SKIPPED, None, "Validation type not yet implemented")
