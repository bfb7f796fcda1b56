"""Reference key-level row verdicts for tg_plan_export_key_rows, built with collections.Counter over the oracle's `_keys`:
uniqueness DUPLICATE / FIRST over the plan table's rows and foreign-key ORPHAN over the child table's rows, each as
(values, validity) lists of bools."""
import math
from collections import Counter

import numpy as np

from oracle import term_oracle as O


def _canon(x):
    # the engine's key equality: -0.0 == +0.0 (Python agrees) and every NaN is one key (Python's NaN objects differ)
    return "NaN" if isinstance(x, float) and math.isnan(x) else x


def _row_keys(table, columns):
    return [tuple(_canon(v) for v in k) for k in O._keys(O.table_cols(table), columns)]


def uniqueness_rows(table, columns):
    """(duplicate, first, validity). One column: a NULL row has no key (invalid); several: a tuple with NULLs is a value."""
    keys = _row_keys(table, columns)
    single = len(columns) == 1
    valid = [not (single and k[0] is None) for k in keys]
    cnt = Counter(k for k, ok in zip(keys, valid) if ok)
    seen, dup, first = set(), [], []
    for k, ok in zip(keys, valid):
        dup.append(ok and cnt[k] >= 2)
        first.append(ok and k not in seen)
        if ok:
            seen.add(k)
    return dup, first, valid


def orphan_rows(tables, child, parent):
    """(orphan, validity) over the child table's rows: a non-NULL child key without a parent; NULL child rows invalid"""
    ct, cc = child.split(".")
    pt, pc = parent.split(".")
    ckeys = [k[0] for k in _row_keys(tables[ct], [cc])]
    pset = {k[0] for k in _row_keys(tables[pt], [pc]) if k[0] is not None}
    valid = [k is not None for k in ckeys]
    return [ok and k not in pset for k, ok in zip(ckeys, valid)], valid


def popcount(values, valid):
    return int(np.count_nonzero(np.asarray(values, dtype=bool) & np.asarray(valid, dtype=bool)))
