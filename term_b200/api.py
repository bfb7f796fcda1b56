"""Host-side mirror of the reference's plugin interface for the hot path (SURVEY.md §8b).

Names, argument meaning and error behaviour follow term-guard so parity tests read like the reference's
own tests:

    ctx = SessionContext()                                   # datafusion::SessionContext (core/context.rs)
    ctx.register_table("data", pyarrow_table)                # MemTable registration
    c = CompletenessConstraint.with_threshold("col", 0.8)    # constraints/completeness.rs:112
    r = c.evaluate(ctx)                                      # Constraint::evaluate (core/constraint.rs:186)
    suite = ValidationSuite.builder("s").check(Check.builder("c").has_size(Assertion.GreaterThan(0)).build()).build()
    suite.run(ctx)                                           # core/suite.rs:399 — here ONE fused GPU plan

Everything numeric happens behind the C ABI (libtermgpu.so); this file only marshals Arrow buffers and
reproduces the orchestration of `ValidationSuite::run_sequential` (core/suite.rs:67-258).
"""
import ctypes as C
import enum
import math
import mmap
import os
import time
from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np

from . import _ffi as F

try:  # pyarrow is the Arrow implementation of the harness; the C ABI itself only sees raw buffers
    import pyarrow as pa
except Exception:  # pragma: no cover
    pa = None


# ----------------------------------------------------------------------------- value types ----
class ConstraintStatus(enum.Enum):  # core/constraint.rs:11-20
    Success = 0
    Failure = 1
    Skipped = 2

    def is_success(self):
        return self is ConstraintStatus.Success

    def is_failure(self):
        return self is ConstraintStatus.Failure

    def is_skipped(self):
        return self is ConstraintStatus.Skipped


@dataclass
class ConstraintResult:  # core/constraint.rs:40-48
    status: ConstraintStatus
    metric: Optional[float] = None
    message: Optional[str] = None
    name: str = ""
    error_code: int = 0


class Assertion:  # constraints/assertion.rs:13-31
    KINDS = ["Equals", "NotEquals", "GreaterThan", "GreaterThanOrEqual", "LessThan", "LessThanOrEqual",
             "Between", "NotBetween"]

    def __init__(self, kind: int, a: float, b: float = 0.0):
        self.kind, self.a, self.b = kind, float(a), float(b)

    def c(self):
        return F.tg_assertion(self.kind, self.a, self.b)

    def evaluate(self, value: float) -> bool:
        return bool(F.lib().tg_assertion_evaluate(self.c(), float(value)))

    def description(self) -> str:
        buf = C.create_string_buffer(256)
        F.lib().tg_assertion_description(self.c(), buf, 256)
        return buf.value.decode()

    def __str__(self):
        return self.description()

    def __repr__(self):
        return f"Assertion.{self.KINDS[self.kind]}({self.a}" + (f", {self.b})" if self.kind >= 6 else ")")


for _i, _n in enumerate(Assertion.KINDS):
    if _i < 6:
        setattr(Assertion, _n, staticmethod(lambda v, _k=_i: Assertion(_k, v)))
    else:
        setattr(Assertion, _n, staticmethod(lambda lo, hi, _k=_i: Assertion(_k, lo, hi)))


class LogicalOperator:  # core/logical.rs:16-27
    def __init__(self, op: int, n: int = 0):
        self.op, self.n = op, n

    def evaluate(self, results: Sequence[bool]) -> bool:
        arr = (C.c_uint8 * max(1, len(results)))(*[1 if r else 0 for r in results])
        return bool(F.lib().tg_logical_evaluate(self.op, self.n, arr, len(results)))

    @staticmethod
    def Exactly(n):
        return LogicalOperator(2, n)

    @staticmethod
    def AtLeast(n):
        return LogicalOperator(3, n)

    @staticmethod
    def AtMost(n):
        return LogicalOperator(4, n)


LogicalOperator.All = LogicalOperator(0)
LogicalOperator.Any = LogicalOperator(1)


class Level(enum.Enum):  # core/level.rs:76-84
    Info = 0
    Warning = 1
    Error = 2


class StatisticType(enum.Enum):  # constraints/statistics.rs:24-45
    Min = 0
    Max = 1
    Mean = 2
    Sum = 3
    StandardDeviation = 4
    Variance = 5
    Median = 6
    Percentile = 7


class FormatType(enum.Enum):  # constraints/format.rs:189-215
    Regex = 0
    Email = 1
    Url = 2
    CreditCard = 3
    Phone = 4
    PostalCode = 5
    UUID = 6
    IPv4 = 7
    IPv6 = 8
    Json = 9
    Iso8601DateTime = 10
    SocialSecurityNumber = 11


@dataclass
class FormatOptions:  # constraints/format.rs:367-480
    case_sensitive: bool = True
    trim_before_check: bool = False
    null_is_valid: bool = True

    @staticmethod
    def strict():
        return FormatOptions(True, False, False)

    @staticmethod
    def lenient():
        return FormatOptions(False, True, True)

    @staticmethod
    def case_insensitive():
        return FormatOptions(False, False, True)

    @staticmethod
    def with_trimming():
        return FormatOptions(True, True, True)


class UniquenessType(enum.Enum):  # constraints/uniqueness.rs:44-60
    FullUniqueness = 0
    Distinctness = 1
    UniqueValueRatio = 2
    PrimaryKey = 3
    UniqueWithNulls = 4
    UniqueComposite = 5


class NullHandling(enum.Enum):
    Exclude = 0
    Include = 1
    Distinct = 2


class CorrelationType(enum.Enum):  # constraints/correlation.rs:20-30 (+ validation kinds)
    Pearson = 0
    Covariance = 1
    Independence = 2
    Spearman = 3
    KendallTau = 4
    MutualInformation = 5
    Range = 6


# ----------------------------------------------------------------------------- context ----
_NP_DTYPES = {np.dtype("int64"): F.TG_INT64, np.dtype("float64"): F.TG_FLOAT64,
              np.dtype("int32"): F.TG_INT32, np.dtype("float32"): F.TG_FLOAT32}


class SessionContext:
    """Owner of registered tables; stands where datafusion's SessionContext stands in the reference."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        F.check(F.lib().tg_engine_create(device, C.byref(self._h)))
        self.device = device
        self._keepalive = {}

    def close(self):
        if self._h:
            F.lib().tg_engine_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def launch_count(self) -> int:
        return int(F.lib().tg_engine_launch_count(self._h))

    def sync_copies(self):
        """tg_engine_sync_copies: pinned host buffers appended from may be freed / reused after this returns"""
        F.check(F.lib().tg_engine_sync_copies(self._h))

    def stream(self) -> int:
        return int(F.lib().tg_engine_stream(self._h) or 0)

    def _create(self, name):
        t = C.c_void_p()
        F.check(F.lib().tg_table_create(self._h, name.encode(), C.byref(t)))
        return t

    def deregister_table(self, name: str):
        F.check(F.lib().tg_table_drop(self._h, name.encode()))
        self._keepalive.pop(name, None)

    def partition_keys(self, table: str, column: str, n_parts: int):
        """tg_table_partition_keys: (device pointer to the valid keys grouped by destination part, keys per part,
        NULL rows). The pointer stays valid until the next partition_keys call on this context."""
        ptr = C.c_void_p()
        counts = (C.c_int64 * n_parts)()
        nulls = C.c_int64()
        F.check(F.lib().tg_table_partition_keys(self._h, table.encode(), column.encode(), n_parts, C.byref(ptr), counts,
                                                C.byref(nulls)))
        return int(ptr.value or 0), [int(c) for c in counts], int(nulls.value)

    def partition_fingerprints(self, table: str, columns, n_parts: int):
        """tg_table_partition_fingerprints: (device pointer to 24-byte {h1, h2, has_null} records grouped by destination
        part, records per part)."""
        ptr = C.c_void_p()
        counts = (C.c_int64 * n_parts)()
        arr, n = _strs(list(columns))
        F.check(F.lib().tg_table_partition_fingerprints(self._h, table.encode(), arr, n, n_parts, C.byref(ptr), counts))
        return int(ptr.value or 0), [int(c) for c in counts]

    def column_dtype(self, table: str, column: str) -> int:
        t = C.c_void_p()
        F.check(F.lib().tg_table_lookup(self._h, table.encode(), C.byref(t)))
        d = C.c_int32()
        F.check(F.lib().tg_table_column_dtype(t, column.encode(), C.byref(d)))
        return int(d.value)

    def column_buffers(self, table: str, column: str) -> dict:
        """tg_table_column_buffers: device addresses of the column's Arrow buffers (engine-owned)"""
        b = F.tg_column_buffers()
        F.check(F.lib().tg_table_column_buffers(self._h, table.encode(), column.encode(), C.byref(b)))
        return {k: getattr(b, k) for k, _ in F.tg_column_buffers._fields_}

    def num_rows(self, name: str) -> int:
        t = C.c_void_p()
        F.check(F.lib().tg_table_lookup(self._h, name.encode(), C.byref(t)))
        return int(F.lib().tg_table_num_rows(t))

    def register_table(self, name: str, data, use_c_data_interface: bool = False):
        """Register host data: a pyarrow Table / RecordBatch / list of RecordBatches, or a dict
        column -> numpy array | (numpy array, validity bool mask) | list of str/None."""
        t = self._create(name)
        try:
            sch = data.schema if pa is not None and isinstance(data, (pa.Table, pa.RecordBatch)) else (
                data[0].schema if isinstance(data, list) and data and pa is not None and isinstance(data[0], pa.RecordBatch) else None)
            if not hasattr(self, "_schemas"):
                self._schemas = {}
            self._schemas[name] = sch
            if pa is not None and isinstance(data, (pa.Table, pa.RecordBatch)):
                batches = data.to_batches() if isinstance(data, pa.Table) else [data]
                if isinstance(data, pa.Table) and not batches:
                    batches = [pa.RecordBatch.from_arrays([pa.array([], type=f.type) for f in data.schema], schema=data.schema)]
                for b in batches:
                    self._append_batch(t, b, use_c_data_interface)
            elif isinstance(data, list) and pa is not None and all(isinstance(b, pa.RecordBatch) for b in data):
                for b in data:
                    self._append_batch(t, b, use_c_data_interface)
            elif isinstance(data, dict):
                arrays = {}
                for col, v in data.items():
                    arrays[col] = _to_arrow(v)
                self._append_batch(t, pa.RecordBatch.from_arrays(list(arrays.values()), names=list(arrays.keys())),
                                   use_c_data_interface)
            else:
                raise TypeError(f"cannot register {type(data)}")
        except Exception:
            F.lib().tg_table_drop(self._h, name.encode())
            raise
        return t

    def _append_batch(self, t, batch, use_c):
        if use_c:
            return self._append_batch_c(t, batch)
        for col_name, arr in zip(batch.schema.names, batch.columns):
            typ = arr.type
            bufs = arr.buffers()
            validity = bufs[0].address if (bufs[0] is not None and arr.null_count > 0) else None
            n, off = len(arr), arr.offset
            if pa.types.is_int64(typ) or pa.types.is_float64(typ) or pa.types.is_int32(typ) or pa.types.is_float32(typ):
                dt = {pa.int64(): F.TG_INT64, pa.float64(): F.TG_FLOAT64, pa.int32(): F.TG_INT32, pa.float32(): F.TG_FLOAT32}[typ]
                w = 8 if dt in (F.TG_INT64, F.TG_FLOAT64) else 4
                vals = (bufs[1].address + off * w) if bufs[1] is not None else None
                F.check(F.lib().tg_table_append_host(t, col_name.encode(), dt, n, vals, None, validity, off))
            elif pa.types.is_string(typ):
                offs = (bufs[1].address + off * 4) if bufs[1] is not None else None
                if offs is None:  # zero-length array without buffers
                    zero = (C.c_int32 * 1)(0)
                    offs = C.addressof(zero)
                vals = bufs[2].address if bufs[2] is not None else None
                F.check(F.lib().tg_table_append_host(t, col_name.encode(), F.TG_UTF8, n, vals, offs, validity, off))
            elif pa.types.is_boolean(typ):
                vals = bufs[1].address if bufs[1] is not None else None
                F.check(F.lib().tg_table_append_host(t, col_name.encode(), F.TG_BOOL, n, vals, None, validity, off))
            else:
                # Int8 .. UInt64, Date / Time / Timestamp / Duration, LargeUtf8: the Arrow C Data Interface entry point widens /
                # narrows them on the host and records the delivered type (DataFusion types MIN / MAX / SUM after it); string
                # dictionaries and string_view arrays (sliced ones too) are decoded to Utf8 on the device; anything it does not
                # know either (decimals, nested types, binary views, non-string dictionaries, ..) raises TG_ERR_UNSUPPORTED
                self._append_batch_c(t, pa.record_batch([arr], names=[col_name]))

    def _append_batch_c(self, t, batch):
        # Arrow C Data Interface: export the batch as a struct array, hand the two structs to the engine
        schema_buf = (C.c_uint8 * 72)()
        array_buf = (C.c_uint8 * 80)()
        batch._export_to_c(C.addressof(array_buf), C.addressof(schema_buf))
        try:
            F.check(F.lib().tg_table_append_arrow(t, C.addressof(schema_buf), C.addressof(array_buf)))
        finally:
            # caller keeps ownership: call the release callbacks (offset 56 in ArrowSchema, 64 in ArrowArray)
            rel_s = C.cast(C.addressof(schema_buf) + 56, C.POINTER(C.c_void_p))[0]
            rel_a = C.cast(C.addressof(array_buf) + 64, C.POINTER(C.c_void_p))[0]
            if rel_a:
                C.CFUNCTYPE(None, C.c_void_p)(rel_a)(C.addressof(array_buf))
            if rel_s:
                C.CFUNCTYPE(None, C.c_void_p)(rel_s)(C.addressof(schema_buf))

    # Parquet physical type -> tg_dtype, decoded on the device (tg_table_append_parquet_chunk)
    # (INT96: the legacy timestamp, stored as Int64 nanoseconds and declared Timestamp(Nanosecond, None) by the engine itself)
    _PARQUET_TYPES = {"INT64": F.TG_INT64, "DOUBLE": F.TG_FLOAT64, "INT32": F.TG_INT32, "FLOAT": F.TG_FLOAT32, "BYTE_ARRAY": F.TG_UTF8,
                      "BOOLEAN": F.TG_BOOL, "INT96": F.TG_PQ_INT96}

    # parquet.thrift CompressionCodec numbers by pyarrow's names: its "LZ4" is the raw block format (thrift LZ4_RAW = 7; the
    # deprecated hadoop-framed thrift LZ4 = 5 reads back as "LZ4_HADOOP")
    _PARQUET_CODECS = {"UNCOMPRESSED": 0, "SNAPPY": 1, "GZIP": 2, "LZO": 3, "BROTLI": 4, "LZ4_HADOOP": 5, "ZSTD": 6, "LZ4": 7, "LZ4_RAW": 7}

    def register_parquet(self, name: str, path, columns=None):
        """ParquetSource::register (sources/parquet.rs:150-230) for the GPU path: every column chunk of every row group
        goes to the engine as raw file bytes (tg_table_append_parquet_chunk) and is decoded into the Arrow layout in HBM.
        The file metadata (row groups, chunk offsets, physical types) is read with pyarrow, like the Rust shim reads it
        with the parquet crate. Unsupported encodings / codecs / types raise: there is no host decode fallback."""
        import pyarrow.parquet as pq
        paths = [path] if isinstance(path, (str, os.PathLike)) else list(path)
        t = self._create(name)
        try:
            return self._register_parquet(t, paths, columns)
        except Exception:
            F.lib().tg_table_drop(self._h, name.encode())  # like register_table: no half-registered table stays behind
            raise

    @staticmethod
    def _check_parquet_logical_type(col, leaf):
        """The device path delivers the PHYSICAL values. Returns the Arrow C-Data format string to declare on the column
        (tg_table_set_column_arrow_type) when the annotation names a type whose Arrow values ARE the physical values — DATE,
        TIME, TIMESTAMP, INT(8|16) — or None for plain columns (unannotated BOOLEAN and INT96 too: the engine declares an INT96
        column Timestamp(Nanosecond, None) itself). Annotations that would need converted values (DECIMAL,
        UINT_32 / UINT_64, raw BYTE_ARRAY) are refused: the reference's ParquetSource yields their logical Arrow types
        (sources/parquet.rs:150-230) and the physical values would be silently wrong."""
        lt = str(getattr(leaf, "logical_type", "NONE") or "NONE").upper()
        ct = str(getattr(leaf, "converted_type", "NONE") or "NONE").upper()
        phys = str(leaf.physical_type)
        if phys == "BYTE_ARRAY":
            # strings only: the string kernels rely on valid UTF-8 (Arrow's Utf8 contract); raw binary is refused
            if lt == "STRING" or ct == "UTF8":
                return None
            raise F.TermGpuError(F.TG_ERR_UNSUPPORTED, f"Parquet column '{col}': BYTE_ARRAY with logical type {lt} / {ct} (only STRING columns)")
        if phys in ("FLOAT", "DOUBLE", "BOOLEAN", "INT96"):
            if lt in ("NONE", "NULL") and ct == "NONE":
                return None
        elif lt in ("NONE", "NULL") and ct in ("NONE", "INT_64", "INT_32"):
            return None
        elif lt.startswith("INT(BITWIDTH=64, ISSIGNED=TRUE") or lt.startswith("INT(BITWIDTH=32, ISSIGNED=TRUE"):
            return None
        elif phys == "INT32" and (lt == "DATE" or ct == "DATE"):
            return "tdD"
        elif phys == "INT32" and lt.startswith("INT(BITWIDTH=8,") or ct in ("INT_8", "UINT_8"):
            return "c" if ("ISSIGNED=TRUE" in lt or ct == "INT_8") else "C"
        elif phys == "INT32" and lt.startswith("INT(BITWIDTH=16,") or ct in ("INT_16", "UINT_16"):
            return "s" if ("ISSIGNED=TRUE" in lt or ct == "INT_16") else "S"
        elif lt.startswith("TIMESTAMP(") and phys == "INT64":
            unit = "m" if "MILLISECONDS" in lt else "u" if "MICROSECONDS" in lt else "n" if "NANOSECONDS" in lt else None
            if unit:
                return f"ts{unit}:" + ("UTC" if "ISADJUSTEDTOUTC=TRUE" in lt else "")
        elif ct in ("TIMESTAMP_MILLIS", "TIMESTAMP_MICROS") and phys == "INT64":
            return "tsm:" if ct == "TIMESTAMP_MILLIS" else "tsu:"
        elif lt.startswith("TIME(") or ct in ("TIME_MILLIS", "TIME_MICROS"):
            if phys == "INT32" and ("MILLISECONDS" in lt or ct == "TIME_MILLIS"):
                return "ttm"
            if phys == "INT64" and ("MICROSECONDS" in lt or ct == "TIME_MICROS"):
                return "ttu"
            if phys == "INT64" and "NANOSECONDS" in lt:
                return "ttn"
        raise F.TermGpuError(F.TG_ERR_UNSUPPORTED, f"Parquet column '{col}': logical type {lt} / {ct} is not decoded on the device "
                                                    "(plain and DATE / TIME / TIMESTAMP / INT(8|16) annotated INT32 / INT64, FLOAT / DOUBLE, BOOLEAN, INT96, STRING)")

    def _register_parquet(self, t, paths, columns):
        import pyarrow.parquet as pq
        declared = {}
        for pth in paths:
            pf = pq.ParquetFile(pth)
            md, schema = pf.metadata, pf.schema
            want = list(columns) if columns is not None else [schema.column(i).name for i in range(md.num_columns)]
            index = {schema.column(i).path: i for i in range(md.num_columns)}
            # the chunks are handed over as views of the mapped file: the only host copy is the engine's staging memcpy
            with open(pth, "rb") as f, mmap.mmap(f.fileno(), 0, flags=mmap.MAP_SHARED | getattr(mmap, "MAP_POPULATE", 0),
                                              prot=mmap.PROT_READ) as mm:  # pre-faulted: no page fault per 4 KB in the staging memcpy
                view = np.frombuffer(mm, dtype=np.uint8)
                try:
                    for rg in range(md.num_row_groups):
                        for col in want:
                            if col not in index:
                                raise F.TermGpuError(2, f"Schema error: No field named {col}.")
                            cm, leaf = md.row_group(rg).column(index[col]), schema.column(index[col])
                            if cm.num_values == 0:
                                continue  # an empty row group holds no pages
                            if cm.physical_type not in self._PARQUET_TYPES:
                                raise F.TermGpuError(F.TG_ERR_UNSUPPORTED, f"Parquet column '{col}': physical type {cm.physical_type} is not decoded on the device")
                            if leaf.max_repetition_level != 0:
                                raise F.TermGpuError(F.TG_ERR_UNSUPPORTED, f"Parquet column '{col}' is repeated")
                            declared[col] = self._check_parquet_logical_type(col, leaf)
                            start = cm.dictionary_page_offset if cm.has_dictionary_page and cm.dictionary_page_offset else cm.data_page_offset
                            chunk = view[start: start + cm.total_compressed_size]
                            codec = self._PARQUET_CODECS.get(cm.compression, 99)  # parquet.thrift CompressionCodec; unknown -> refused
                            F.check(F.lib().tg_table_append_parquet_chunk(t, col.encode(), self._PARQUET_TYPES[cm.physical_type],
                                                                          leaf.max_definition_level, codec, chunk.ctypes.data,
                                                                          chunk.size, cm.num_values))
                finally:
                    chunk = None
                    del view  # the mapping cannot close while a buffer export is alive
        for col, fmt in declared.items():
            if fmt is not None:
                F.check(F.lib().tg_table_set_column_arrow_type(t, col.encode(), fmt.encode()))
        return t

    def register_csv(self, name: str, path, schema, has_header: bool = True, delimiter: str = ",", quote: str = '"', escape: Optional[str] = None,
                     comment: Optional[str] = None, terminator: Optional[str] = None, null_regex: Optional[str] = None):
        """CsvSource::register for the GPU path: the file is mapped and tokenized / parsed into the Arrow layout in HBM
        (tg_table_append_csv_format), with `schema` (a pyarrow.Schema, in file order) giving every column's name and type. Schema
        inference is not done here: DataFusion infers with arrow-csv's rules, which the Rust shim would call on the host.
        quote / escape / comment / terminator (one byte each; None: no escape, no comment, records end at LF, CRLF or CR) and
        null_regex (None: an empty field is NULL) are CsvReadOptions' fields of the same names (include/termgpu.h states the rules).
        Unsupported types and malformed records raise; no half-registered table stays behind."""
        if pa is None or not isinstance(schema, pa.Schema):
            raise TypeError("register_csv needs a pyarrow.Schema")
        fmt = csv_format(delimiter, quote, escape, comment, terminator, null_regex, has_header)
        names, fmts = _strs([f.name for f in schema]), _strs([_arrow_format(f.type) for f in schema])
        t = self._create(name)
        try:
            with open(path, "rb") as f:
                size = os.fstat(f.fileno()).st_size
                rows = C.c_int64()
                if size == 0:
                    F.check(F.lib().tg_table_append_csv_format(t, names[0], fmts[0], len(schema), None, 0, C.byref(fmt), C.byref(rows)))
                else:
                    with mmap.mmap(f.fileno(), 0, flags=mmap.MAP_SHARED | getattr(mmap, "MAP_POPULATE", 0), prot=mmap.PROT_READ) as mm:
                        view = np.frombuffer(mm, dtype=np.uint8)
                        try:
                            F.check(F.lib().tg_table_append_csv_format(t, names[0], fmts[0], len(schema), view.ctypes.data, size, C.byref(fmt),
                                                                       C.byref(rows)))
                        finally:
                            del view  # the mapping cannot close while a buffer export is alive
        except Exception:
            F.lib().tg_table_drop(self._h, name.encode())
            raise
        if not hasattr(self, "_schemas"):
            self._schemas = {}
        self._schemas[name] = schema
        return t

    def register_arrow_device(self, name: str, data):
        """Register RecordBatches through the Arrow C Device Data Interface: `data` is one object implementing
        `__arrow_c_device_array__` (a RecordBatch; CUDA, CUDA_MANAGED, CUDA_HOST or CPU memory) or a list of them, each one
        tg_table_append_arrow_device call. CUDA batches are converted in HBM; the producer may free or reuse its buffers as
        soon as this returns. A failed append drops the table, as register_table does."""
        if pa is None:
            raise TypeError("register_arrow_device needs pyarrow")
        batches = list(data) if isinstance(data, (list, tuple)) else [data]
        t = self._create(name)
        schema = None
        try:
            for b in batches:
                sc, ac = b.__arrow_c_device_array__()
                F.check(F.lib().tg_table_append_arrow_device(t, _capsule_pointer(sc, b"arrow_schema"), _capsule_pointer(ac, b"arrow_device_array")))
                if schema is None:
                    schema = pa.Schema._import_from_c_capsule(sc)
        except Exception:
            F.lib().tg_table_drop(self._h, name.encode())
            raise
        if not hasattr(self, "_schemas"):
            self._schemas = {}
        self._schemas[name] = schema
        return t

    def register_device_table(self, name: str, columns: Dict[str, dict], keepalive=None):
        """Adopt HBM-resident Arrow buffers without copying. columns[name] = dict(dtype=TG_*, n_rows=,
        values=ptr, validity=ptr|None, offsets=ptr|None, n_value_bytes=int). Pointers are device addresses."""
        t = self._create(name)
        for col, d in columns.items():
            F.check(F.lib().tg_table_adopt_device(t, col.encode(), d["dtype"], d["n_rows"], d.get("values"),
                                                  d.get("offsets"), d.get("validity"), d.get("n_value_bytes", 0)))
        self._keepalive[name] = keepalive
        return t


def _capsule_pointer(capsule, name: bytes) -> int:
    get = C.pythonapi.PyCapsule_GetPointer
    get.restype, get.argtypes = C.c_void_p, [C.py_object, C.c_char_p]
    return get(capsule, name)


def _to_arrow(v):
    if pa is not None and isinstance(v, (pa.Array, pa.ChunkedArray)):
        return v.combine_chunks() if isinstance(v, pa.ChunkedArray) else v
    if isinstance(v, tuple):
        vals, mask = v
        return pa.array(np.asarray(vals), mask=~np.asarray(mask, dtype=bool))
    if isinstance(v, np.ndarray):
        return pa.array(v)
    return pa.array(v)


# ----------------------------------------------------------------------------- plan ----
class Plan:
    """Thin RAII wrapper of tg_plan."""

    def __init__(self):
        self._h = C.c_void_p()
        F.check(F.lib().tg_plan_create(C.byref(self._h)))

    def __del__(self):
        try:
            if self._h:
                F.lib().tg_plan_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def execute(self, ctx: SessionContext, table: str = "data"):
        self._ctx_schema = getattr(ctx, "_schemas", {}).get(table)  # (schema-only constraints read it, as the reference reads df.schema())
        self._ctx = ctx  # (constraints that name their own table — TemporalOrderingConstraint — evaluate against it from _result)
        F.check(F.lib().tg_plan_execute(ctx.handle, self._h, table.encode()))

    def execute_partial(self, ctx: SessionContext, table: str = "data"):
        self._ctx_schema = getattr(ctx, "_schemas", {}).get(table)
        self._ctx = ctx
        F.check(F.lib().tg_plan_execute_partial(ctx.handle, self._h, table.encode()))

    def partial_export(self) -> bytes:
        n = C.c_size_t()
        F.check(F.lib().tg_plan_partial_size(self._h, C.byref(n)))
        buf = C.create_string_buffer(n.value)
        F.check(F.lib().tg_plan_partial_export(self._h, buf, n.value))
        return buf.raw

    def partial_reset(self):
        F.check(F.lib().tg_plan_partial_reset(self._h))

    def partial_merge(self, blob: bytes):
        F.check(F.lib().tg_plan_partial_merge(self._h, blob, len(blob)))

    def finalize(self):
        F.check(F.lib().tg_plan_finalize(self._h))

    def set_aggregate_partial(self, agg_index: int, u, f):
        """tg_plan_set_aggregate_partial: install an externally computed partial state (distributed Spearman)"""
        uu = (C.c_uint64 * 8)(*[int(x) for x in u])
        ff = (C.c_double * 8)(*[float(x) for x in f])
        F.check(F.lib().tg_plan_set_aggregate_partial(self._h, agg_index, uu, ff))

    def kll_levels(self, slot: int):
        """the slot's sketch as KllSketch's compactor stack: [items of level 0, items of level 1, ..] (weight 2^level)"""
        nl = F.check_slot(F.lib().tg_plan_kll_levels(self._h, slot, -1, None, 0))
        out = []
        for lv in range(nl):
            c = F.check_slot(F.lib().tg_plan_kll_levels(self._h, slot, lv, None, 0))
            buf = (C.c_double * max(c, 1))()
            F.check_slot(F.lib().tg_plan_kll_levels(self._h, slot, lv, buf, c))
            out.append(list(buf[:c]))
        return out

    def histogram_pending(self):
        """indices of HIST aggregates whose merged shards disagreed on [min, max] (second phase needed)"""
        n = F.check_slot(F.lib().tg_plan_histogram_pending(self._h, None, 0))
        if n == 0:
            return []
        idx = (C.c_int32 * n)()
        F.check_slot(F.lib().tg_plan_histogram_pending(self._h, idx, n))
        return list(idx)

    def _hist_buckets(self, agg_index: int) -> int:
        return int(self.aggregates()[agg_index][1].split("|")[-1])

    def histogram_rebucket(self, ctx: "SessionContext", table: str, agg_index: int):
        """this shard's bucket counts against the merged (global) min / max"""
        nb = self._hist_buckets(agg_index)
        counts = (C.c_uint64 * nb)()
        F.check(F.lib().tg_plan_histogram_rebucket(ctx.handle, self._h, table.encode(), agg_index, counts, nb))
        return list(counts)

    def histogram_install(self, agg_index: int, counts):
        nb = len(counts)
        arr = (C.c_uint64 * nb)(*counts)
        F.check(F.lib().tg_plan_histogram_install(self._h, agg_index, arr, nb))

    def redirect(self, agg_index: int, which: int, table):
        """tg_plan_redirect_aggregate: aggregate `agg_index` reads its keys from `table` (None: undo)."""
        F.check(F.lib().tg_plan_redirect_aggregate(self._h, agg_index, which, table.encode() if table else None))

    def aggregates(self):
        """[(kind, key)] of the plan's device aggregates, in partial-blob order."""
        n = F.lib().tg_plan_num_aggregates(self._h)
        cached = getattr(self, "_aggs_cache", None)
        if cached is not None and len(cached) == n:  # aggregates are only ever appended
            return cached
        out = []
        for i in range(n):
            k, key = C.c_int32(), C.c_char_p()
            F.check(F.lib().tg_plan_aggregate_info(self._h, i, C.byref(k), C.byref(key)))
            out.append((k.value, key.value.decode()))
        self._aggs_cache = out
        return out

    def result(self, slot: int) -> ConstraintResult:
        r = F.tg_result()
        F.check(F.lib().tg_plan_result(self._h, slot, C.byref(r)))
        return ConstraintResult(ConstraintStatus(r.status), r.metric if r.has_metric else None,
                                r.message.decode("utf-8", "replace") if r.message else None,
                                r.name.decode() if r.name else "", r.error_code)

    def analyzer_result(self, slot: int):
        r = F.tg_analyzer_result()
        F.check(F.lib().tg_plan_analyzer_result(self._h, slot, C.byref(r)))
        m = {}
        n = F.lib().tg_plan_map_size(self._h, slot)
        for i in range(max(n, 0)):
            k, v = C.c_char_p(), C.c_double()
            F.check(F.lib().tg_plan_map_entry(self._h, slot, i, C.byref(k), C.byref(v)))
            m[k.value.decode()] = v.value
        return AnalyzerOutput(list(r.u), list(r.f), r.metric_kind, r.error, r.metric_double, r.metric_long,
                              r.metric_key.decode() if r.metric_key else "",
                              r.message.decode("utf-8", "replace") if r.message else None, m)

    def analyzer_state_json(self, slot: int) -> str:
        """serde_json text of the slot's *State struct (FileSystemStateStore format); "" when it has none"""
        n = F.check_slot(F.lib().tg_plan_analyzer_state_json(self._h, slot, None, 0))
        buf = C.create_string_buffer(n + 1)
        F.check_slot(F.lib().tg_plan_analyzer_state_json(self._h, slot, buf, n + 1))
        return buf.value.decode()

    def stats(self):
        s = F.tg_exec_stats()
        F.check(F.lib().tg_plan_exec_stats(self._h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in F.tg_exec_stats._fields_}


@dataclass
class AnalyzerOutput:
    u: List[int]
    f: List[float]
    metric_kind: int   # 0 Double, 1 Long, 2 Map, 3 none
    error: int         # 0 ok, 1 NoData, 2 InvalidData
    metric_double: float
    metric_long: int
    metric_key: str
    message: Optional[str]
    map: Dict[str, float]

    @property
    def metric(self):
        if self.error:
            return None
        return {0: self.metric_double, 1: self.metric_long, 2: self.map}.get(self.metric_kind)


def csv_format(delimiter=",", quote='"', escape=None, comment=None, terminator=None, null_regex=None, has_header=True):
    """a tg_csv_format from register_csv's options (each byte option one byte, as str or bytes; None: the default)"""
    def byte(what, v):
        if v is None:
            return -1
        b = v.encode() if isinstance(v, str) else bytes(v)
        if len(b) != 1:
            raise ValueError(f"the {what} must be one byte")
        return b[0]
    if delimiter is None or quote is None:
        raise ValueError("the delimiter and the quote must be one byte")
    rx = null_regex.encode() if isinstance(null_regex, str) else null_regex
    return F.tg_csv_format(byte("delimiter", delimiter), byte("quote", quote), byte("escape", escape), byte("comment", comment),
                           byte("terminator", terminator), int(has_header), rx)


def _arrow_format(typ):
    """the Arrow C Data Interface format string of a pyarrow type (what tg_table_append_csv takes)"""
    schema_buf = (C.c_uint8 * 72)()
    typ._export_to_c(C.addressof(schema_buf))
    try:
        return C.cast(C.cast(C.addressof(schema_buf), C.POINTER(C.c_void_p))[0], C.c_char_p).value.decode()
    finally:
        rel = C.cast(C.addressof(schema_buf) + 56, C.POINTER(C.c_void_p))[0]
        if rel:
            C.CFUNCTYPE(None, C.c_void_p)(rel)(C.addressof(schema_buf))


def _strs(cols):
    arr = (C.c_char_p * max(1, len(cols)))(*[c.encode() for c in cols])
    return arr, len(cols)


def _opt(s):
    return s.encode() if s is not None else None


# ----------------------------------------------------------------------------- constraints ----
class Constraint:
    """core/constraint.rs:186-225 — evaluate(ctx) -> ConstraintResult; name(); column()."""

    def _add_to(self, plan: Plan) -> int:
        raise NotImplementedError

    def _result(self, plan: Plan, slot: int) -> ConstraintResult:
        """the slot's result; constraints whose assertion is a host closure (HistogramConstraint) finish it here"""
        return plan.result(slot)

    def evaluate(self, ctx: SessionContext, table: str = "data") -> ConstraintResult:
        plan = Plan()
        slot = self._add_to(plan)
        plan.execute(ctx, table)
        return self._result(plan, slot)

    def name(self):
        plan = Plan()
        slot = self._add_to(plan)
        plan.finalize()
        return plan.result(slot).name


class CompletenessConstraint(Constraint):  # constraints/completeness.rs
    def __init__(self, columns, threshold=1.0, operator=None):
        self.columns = [columns] if isinstance(columns, str) else list(columns)
        self.threshold = threshold
        self.operator = operator or LogicalOperator.All
        self._validate()

    def _validate(self):
        self._add_to(Plan())

    @staticmethod
    def with_threshold(columns, threshold):
        return CompletenessConstraint(columns, threshold)

    @staticmethod
    def complete(columns):
        return CompletenessConstraint(columns, 1.0)

    @staticmethod
    def with_operator(columns, operator, threshold):
        return CompletenessConstraint(columns, threshold, operator)

    def _add_to(self, plan):
        arr, n = _strs(self.columns)
        return F.check_slot(F.lib().tg_plan_add_completeness(plan.handle, arr, n, self.threshold,
                                                             self.operator.op, self.operator.n))


class SizeConstraint(Constraint):  # constraints/size.rs
    def __init__(self, assertion: Assertion):
        self.assertion = assertion

    def _add_to(self, plan):
        return F.check_slot(F.lib().tg_plan_add_size(plan.handle, self.assertion.c()))


class LengthAssertion:  # constraints/length.rs:20-60
    """LengthAssertion::{Min, Max, Between, Exactly, NotEmpty}"""
    def __init__(self, kind, a=0, b=0):
        self.kind, self.a, self.b = kind, a, b

    @staticmethod
    def Min(n): return LengthAssertion(0, n)
    @staticmethod
    def Max(n): return LengthAssertion(1, n)
    @staticmethod
    def Between(a, b): return LengthAssertion(2, a, b)
    @staticmethod
    def Exactly(n): return LengthAssertion(3, n)
    @staticmethod
    def NotEmpty(): return LengthAssertion(4)


class LengthConstraint(Constraint):  # constraints/length.rs:86-232
    def __init__(self, column, assertion: LengthAssertion):
        self.column, self.assertion = column, assertion
        self._add_to(Plan())

    @staticmethod
    def min(c, n): return LengthConstraint(c, LengthAssertion.Min(n))
    @staticmethod
    def max(c, n): return LengthConstraint(c, LengthAssertion.Max(n))
    @staticmethod
    def between(c, a, b): return LengthConstraint(c, LengthAssertion.Between(a, b))
    @staticmethod
    def exactly(c, n): return LengthConstraint(c, LengthAssertion.Exactly(n))
    @staticmethod
    def not_empty(c): return LengthConstraint(c, LengthAssertion.NotEmpty())

    def _add_to(self, plan):
        a = self.assertion
        return F.check_slot(F.lib().tg_plan_add_length(plan.handle, self.column.encode(), a.kind, a.a, a.b))


class ContainmentConstraint(Constraint):  # constraints/values.rs:205-331
    def __init__(self, column, allowed_values):
        self.column, self.allowed_values = column, [str(v) for v in allowed_values]
        self._add_to(Plan())

    def _add_to(self, plan):
        arr = (C.c_char_p * max(1, len(self.allowed_values)))(*[v.encode() for v in self.allowed_values])
        return F.check_slot(F.lib().tg_plan_add_containment(plan.handle, self.column.encode(), arr, len(self.allowed_values)))


class NonNegativeConstraint(Constraint):  # constraints/values.rs:336-440
    def __init__(self, column):
        self.column = column
        self._add_to(Plan())

    def _add_to(self, plan):
        return F.check_slot(F.lib().tg_plan_add_non_negative(plan.handle, self.column.encode()))


class ApproxCountDistinctConstraint(Constraint):  # constraints/approx_count_distinct.rs
    def __init__(self, column, assertion: Assertion):
        self.column, self.assertion = column, assertion
        self._add_to(Plan())

    def _add_to(self, plan):
        return F.check_slot(F.lib().tg_plan_add_approx_count_distinct(plan.handle, self.column.encode(), self.assertion.c()))


class DataType(enum.IntEnum):  # constraints/values.rs:14-26
    Integer = 0
    Float = 1
    Boolean = 2
    Date = 3
    Timestamp = 4
    String = 5


class DataTypeConstraint(Constraint):  # constraints/values.rs:69-196
    def __init__(self, column, data_type: DataType, threshold: float):
        self.column, self.data_type, self.threshold = column, data_type, threshold
        self._add_to(Plan())

    def _add_to(self, plan):
        return F.check_slot(F.lib().tg_plan_add_data_type(plan.handle, self.column.encode(), int(self.data_type), float(self.threshold)))


class ColumnCountConstraint(Constraint):  # constraints/column_count.rs
    def __init__(self, assertion: Assertion):
        self.assertion = assertion

    def _add_to(self, plan):
        return F.check_slot(F.lib().tg_plan_add_column_count(plan.handle, self.assertion.c()))


class StatisticalConstraint(Constraint):  # constraints/statistics.rs:120-322
    def __init__(self, column, statistic: StatisticType, assertion: Assertion, percentile: float = 0.0):
        self.column, self.statistic, self.assertion, self.percentile = column, statistic, assertion, percentile
        self._add_to(Plan())

    @staticmethod
    def min(c, a): return StatisticalConstraint(c, StatisticType.Min, a)
    @staticmethod
    def max(c, a): return StatisticalConstraint(c, StatisticType.Max, a)
    @staticmethod
    def mean(c, a): return StatisticalConstraint(c, StatisticType.Mean, a)
    @staticmethod
    def sum(c, a): return StatisticalConstraint(c, StatisticType.Sum, a)
    @staticmethod
    def standard_deviation(c, a): return StatisticalConstraint(c, StatisticType.StandardDeviation, a)
    @staticmethod
    def variance(c, a): return StatisticalConstraint(c, StatisticType.Variance, a)
    @staticmethod
    def median(c, a): return StatisticalConstraint(c, StatisticType.Median, a)
    @staticmethod
    def percentile_(c, p, a): return StatisticalConstraint(c, StatisticType.Percentile, a, p)

    def _add_to(self, plan):
        return F.check_slot(F.lib().tg_plan_add_statistic(plan.handle, self.column.encode(), self.statistic.value,
                                                          self.percentile, self.assertion.c()))


class MultiStatisticalConstraint(Constraint):  # constraints/statistics.rs:385-504
    def __init__(self, column, statistics):
        self.column, self.statistics = column, list(statistics)
        self._add_to(Plan())

    def _add_to(self, plan):
        n = len(self.statistics)
        kinds = (C.c_int32 * max(1, n))(*[s[0].value if isinstance(s[0], StatisticType) else s[0][0].value for s in self.statistics])
        pcts = (C.c_double * max(1, n))(*[0.0 if isinstance(s[0], StatisticType) else s[0][1] for s in self.statistics])
        asr = (F.tg_assertion * max(1, n))(*[s[1].c() for s in self.statistics])
        return F.check_slot(F.lib().tg_plan_add_multi_statistic(plan.handle, self.column.encode(), kinds, pcts, asr, n))


@dataclass
class QuantileCheck:  # constraints/quantile.rs:38-58
    quantile: float
    assertion: Assertion

    def __post_init__(self):
        if not (0.0 <= self.quantile <= 1.0):
            raise F.TermGpuError(F.TG_ERR_CONFIGURATION, "Quantile must be between 0.0 and 1.0")


class QuantileConstraint(Constraint):  # constraints/quantile.rs:147-497
    """QuantileValidation: Single / Multiple / Monotonic evaluate; Distribution / Custom are Skipped like the
    reference's catch-all arm (:474-479). Every quantile of a column shares the plan's one KLL sketch."""
    SINGLE, MULTIPLE, MONOTONIC, UNIMPLEMENTED = 0, 1, 2, 3

    def __init__(self, column, validation, checks=(), quantiles=(), strict=False):
        self.column, self.validation, self.strict = column, validation, strict
        self.checks, self.quantiles = list(checks), list(quantiles)
        self._add_to(Plan())

    @staticmethod
    def median(column, assertion): return QuantileConstraint.percentile(column, 0.5, assertion)
    @staticmethod
    def percentile(column, q, assertion): return QuantileConstraint(column, QuantileConstraint.SINGLE, [QuantileCheck(q, assertion)])
    @staticmethod
    def multiple(column, checks): return QuantileConstraint(column, QuantileConstraint.MULTIPLE, checks)
    @staticmethod
    def monotonic(column, quantiles, strict): return QuantileConstraint(column, QuantileConstraint.MONOTONIC, quantiles=quantiles, strict=strict)
    @staticmethod
    def distribution(column, config=None): return QuantileConstraint(column, QuantileConstraint.UNIMPLEMENTED)

    def _add_to(self, plan):
        qs = [c.quantile for c in self.checks] if self.checks else self.quantiles
        n = len(qs)
        q = (C.c_double * max(1, n))(*qs)
        asr = (F.tg_assertion * max(1, n))(*[c.assertion.c() for c in self.checks]) if self.checks else None
        return F.check_slot(F.lib().tg_plan_add_quantile(plan.handle, self.column.encode(), self.validation, q, asr,
                                                         n, int(self.strict)))


class FormatConstraint(Constraint):  # constraints/format.rs:482-843
    def __init__(self, column, format: FormatType, threshold, options: FormatOptions = None, arg=None, flag=False):
        self.column, self.format, self.threshold = column, format, threshold
        self.options = options or FormatOptions()
        self.arg, self.flag = arg, flag
        self._add_to(Plan())

    @staticmethod
    def new(column, format, threshold, options, arg=None, flag=False):
        return FormatConstraint(column, format, threshold, options, arg, flag)

    @staticmethod
    def email(c, t): return FormatConstraint(c, FormatType.Email, t)
    @staticmethod
    def url(c, t, allow_localhost): return FormatConstraint(c, FormatType.Url, t, flag=allow_localhost)
    @staticmethod
    def credit_card(c, t, detect_only): return FormatConstraint(c, FormatType.CreditCard, t, flag=detect_only)
    @staticmethod
    def phone(c, t, country=None): return FormatConstraint(c, FormatType.Phone, t, FormatOptions(trim_before_check=True), arg=country)
    @staticmethod
    def postal_code(c, t, country): return FormatConstraint(c, FormatType.PostalCode, t, FormatOptions(trim_before_check=True), arg=country)
    @staticmethod
    def uuid(c, t): return FormatConstraint(c, FormatType.UUID, t)
    @staticmethod
    def ipv4(c, t): return FormatConstraint(c, FormatType.IPv4, t)
    @staticmethod
    def ipv6(c, t): return FormatConstraint(c, FormatType.IPv6, t)
    @staticmethod
    def json(c, t): return FormatConstraint(c, FormatType.Json, t)
    @staticmethod
    def iso8601_datetime(c, t): return FormatConstraint(c, FormatType.Iso8601DateTime, t)
    @staticmethod
    def regex(c, pattern, t): return FormatConstraint(c, FormatType.Regex, t, arg=pattern)
    @staticmethod
    def social_security_number(c, t): return FormatConstraint(c, FormatType.SocialSecurityNumber, t, FormatOptions(trim_before_check=True))

    def _add_to(self, plan):
        o = F.tg_format_options(int(self.options.case_sensitive), int(self.options.trim_before_check),
                                int(self.options.null_is_valid))
        return F.check_slot(F.lib().tg_plan_add_format(plan.handle, self.column.encode(), self.format.value,
                                                       _opt(self.arg), int(bool(self.flag)), self.threshold, C.byref(o)))


class UniquenessConstraint(Constraint):  # constraints/uniqueness.rs
    def __init__(self, columns, uniqueness_type: UniquenessType, threshold=1.0, assertion: Assertion = None,
                 null_handling: NullHandling = NullHandling.Exclude):
        self.columns = [columns] if isinstance(columns, str) else list(columns)
        self.uniqueness_type, self.threshold = uniqueness_type, threshold
        self.assertion = assertion or Assertion.Equals(0.0)
        self.null_handling = null_handling
        self._add_to(Plan())

    @staticmethod
    def full_uniqueness(column, threshold): return UniquenessConstraint([column], UniquenessType.FullUniqueness, threshold)
    @staticmethod
    def full_uniqueness_multi(columns, threshold): return UniquenessConstraint(columns, UniquenessType.FullUniqueness, threshold)
    @staticmethod
    def distinctness(columns, assertion): return UniquenessConstraint(columns, UniquenessType.Distinctness, assertion=assertion)
    @staticmethod
    def unique_value_ratio(columns, assertion): return UniquenessConstraint(columns, UniquenessType.UniqueValueRatio, assertion=assertion)
    @staticmethod
    def primary_key(columns): return UniquenessConstraint(columns, UniquenessType.PrimaryKey)
    @staticmethod
    def unique_with_nulls(columns, threshold, null_handling): return UniquenessConstraint(columns, UniquenessType.UniqueWithNulls, threshold, null_handling=null_handling)
    @staticmethod
    def unique_composite(columns, threshold, null_handling, case_sensitive=True): return UniquenessConstraint(columns, UniquenessType.UniqueComposite, threshold, null_handling=null_handling)

    def column(self):
        return self.columns[0] if len(self.columns) == 1 else None

    def _add_to(self, plan):
        arr, n = _strs(self.columns)
        return F.check_slot(F.lib().tg_plan_add_uniqueness(plan.handle, arr, n, self.uniqueness_type.value,
                                                           self.threshold, self.assertion.c(), self.null_handling.value))


class CorrelationConstraint(Constraint):  # constraints/correlation.rs
    def __init__(self, column1, column2, kind: CorrelationType, assertion: Assertion):
        self.column1, self.column2, self.kind, self.assertion = column1, column2, kind, assertion
        self._add_to(Plan())

    @staticmethod
    def pearson(c1, c2, assertion): return CorrelationConstraint(c1, c2, CorrelationType.Pearson, assertion)
    @staticmethod
    def spearman(c1, c2, assertion): return CorrelationConstraint(c1, c2, CorrelationType.Spearman, assertion)
    @staticmethod
    def covariance(c1, c2, assertion): return CorrelationConstraint(c1, c2, CorrelationType.Covariance, assertion)
    @staticmethod
    def independence(c1, c2, max_correlation): return CorrelationConstraint(c1, c2, CorrelationType.Independence, Assertion(0, max_correlation))
    @staticmethod
    def correlation_range(c1, c2, lo, hi): return CorrelationConstraint(c1, c2, CorrelationType.Range, Assertion.Between(lo, hi))

    def _add_to(self, plan):
        return F.check_slot(F.lib().tg_plan_add_correlation(plan.handle, self.column1.encode(), self.column2.encode(),
                                                            self.kind.value, self.assertion.c()))


class CustomSqlConstraint(Constraint):  # constraints/custom_sql.rs
    def __init__(self, expression: str, hint: Optional[str] = None):
        self.expression, self.hint = expression, hint
        self._add_to(Plan())

    def _add_to(self, plan):
        return F.check_slot(F.lib().tg_plan_add_custom_sql(plan.handle, self.expression.encode(), _opt(self.hint)))


class ForeignKeyConstraint(Constraint):  # constraints/foreign_key.rs
    def __init__(self, child_column: str, parent_column: str):
        self.child_column, self.parent_column = child_column, parent_column
        self._allow_nulls, self._max = False, 100

    def allow_nulls(self, allow: bool):
        self._allow_nulls = allow
        return self

    def max_violations_reported(self, n: int):
        self._max = n
        return self

    def _add_to(self, plan):
        return F.check_slot(F.lib().tg_plan_add_foreign_key(plan.handle, self.child_column.encode(),
                                                            self.parent_column.encode(), int(self._allow_nulls), self._max))


# ----------------------------------------------------------------------------- Check / Suite ----
@dataclass
class HistogramBucket:  # constraints/histogram.rs:14-22
    value: str
    count: int
    ratio: float


class Histogram:  # constraints/histogram.rs:25-127
    def __init__(self, buckets, total_count, null_count):
        self.buckets, self.total_count, self.null_count = list(buckets), total_count, null_count
        self.distinct_count = len(self.buckets)

    def most_common_ratio(self): return self.buckets[0].ratio if self.buckets else 0.0
    def least_common_ratio(self): return self.buckets[-1].ratio if self.buckets else 0.0
    def bucket_count(self): return len(self.buckets)
    def top_n(self, n): return [(b.value, b.ratio) for b in self.buckets[:n]]

    def is_roughly_uniform(self, threshold):
        if not self.buckets:
            return True
        lo = self.least_common_ratio()
        return False if lo == 0.0 else self.most_common_ratio() / lo <= threshold

    def get_value_ratio(self, value):
        return next((b.ratio for b in self.buckets if b.value == value), None)

    def entropy(self):
        e = 0.0
        for b in self.buckets:
            if b.ratio > 0.0:
                e += -b.ratio * math.log(b.ratio)
        return e

    def follows_power_law(self, top_n, threshold):
        s = 0.0
        for b in self.buckets[:top_n]:
            s += b.ratio
        return s >= threshold

    def null_ratio(self): return 0.0 if self.total_count == 0 else self.null_count / self.total_count


class HistogramConstraint(Constraint):  # constraints/histogram.rs:129-413
    """The value frequencies come from the GPU (tg_plan_add_value_histogram: the grouped-count kernel over the column itself);
    the assertion is a host closure over the Histogram, as in the reference."""

    def __init__(self, column, assertion: Callable[[Histogram], bool], description="custom assertion"):
        self.column, self.assertion, self.assertion_description = column, assertion, description

    @staticmethod
    def new_with_description(column, assertion, description): return HistogramConstraint(column, assertion, description)

    def _add_to(self, plan):
        return F.check_slot(F.lib().tg_plan_add_value_histogram(plan.handle, self.column.encode()))

    def histogram(self, plan, slot) -> Histogram:
        a = plan.analyzer_result(slot)
        total, nulls = a.u[0], a.u[1]
        return Histogram([HistogramBucket(k, int(v), int(v) * 1.0 / (total - nulls)) for k, v in a.map.items()], total, nulls)

    def _result(self, plan, slot):
        r = plan.result(slot)
        if r.status is not ConstraintStatus.Success:  # Skipped("No data to analyze") / an evaluation error
            return r
        h = self.histogram(plan, slot)
        if self.assertion(h):
            return r
        r.status = ConstraintStatus.Failure
        r.message = (f"Histogram assertion '{self.assertion_description}' failed for column '{self.column}'. Distribution: {h.distinct_count} "
                     f"distinct values, most common ratio: {h.most_common_ratio() * 100.0:.2f}%, null ratio: {h.null_ratio() * 100.0:.2f}%")
        return r


def arrow_type_debug(t) -> str:
    """`{:?}` of the arrow-rs DataType a pyarrow type corresponds to (what DataTypeConstraint::specific_type compares with)"""
    simple = {"int8": "Int8", "int16": "Int16", "int32": "Int32", "int64": "Int64", "uint8": "UInt8", "uint16": "UInt16", "uint32": "UInt32",
              "uint64": "UInt64", "float": "Float32", "double": "Float64", "halffloat": "Float16", "bool": "Boolean", "string": "Utf8",
              "large_string": "LargeUtf8", "binary": "Binary", "large_binary": "LargeBinary", "date32[day]": "Date32", "date64[ms]": "Date64", "null": "Null",
              "string_view": "Utf8View", "binary_view": "BinaryView"}
    k = str(t)
    if k in simple:
        return simple[k]
    if pa.types.is_dictionary(t):
        return f"Dictionary({arrow_type_debug(t.index_type)}, {arrow_type_debug(t.value_type)})"
    units = {"s": "Second", "ms": "Millisecond", "us": "Microsecond", "ns": "Nanosecond"}
    if pa.types.is_timestamp(t):
        return f"Timestamp({units[t.unit]}, " + ("None" if t.tz is None else f'Some("{t.tz}")') + ")"
    if pa.types.is_duration(t):
        return f"Duration({units[t.unit]})"
    if pa.types.is_time(t):
        return f"Time{t.bit_width}({units[t.unit]})"
    return k


class UnifiedDataTypeConstraint(Constraint):  # constraints/datatype.rs:236-445 (the reference's second DataTypeConstraint)
    """SpecificType reads the schema; Consistency is the reference's placeholder (column must exist, consistency = 0.95);
    every other validation is a predicate counted over the non-NULL rows — here the non-NULL count (K1 validity popcount)
    and the count of rows where `col IS NOT NULL AND (predicate)` holds (K1 predicate unit), fused into one scan."""

    def __init__(self, column, kind, predicate=None, description="", threshold=None, expected=None):
        F.check(F.lib().tg_validate_identifier(column.encode()))
        if kind == "consistency" and not (0.0 <= threshold <= 1.0):
            raise ValueError("Threshold must be between 0.0 and 1.0")
        self.column, self.kind, self.predicate, self.description, self.threshold, self.expected = column, kind, predicate, description, threshold, expected

    @staticmethod
    def _esc(column): return '"' + column.replace('"', '""') + '"'

    @classmethod
    def specific_type(cls, column, data_type): return cls(column, "specific", expected=data_type, description=f"type is {data_type}")
    @classmethod
    def type_consistency(cls, column, threshold): return cls(column, "consistency", threshold=threshold)
    @classmethod
    def _pred(cls, column, template, description): return cls(column, "predicate", template.replace("{c}", cls._esc(column)), description)
    @classmethod
    def non_negative(cls, column): return cls._pred(column, "{c} >= 0", "non-negative values")
    @classmethod
    def positive(cls, column): return cls._pred(column, "{c} > 0", "positive values")
    @classmethod
    def integer(cls, column): return cls._pred(column, "{c} = CAST({c} AS INT)", "integer values")
    @classmethod
    def range(cls, column, lo, hi): return cls._pred(column, "{c} BETWEEN " + _rust_num(lo) + " AND " + _rust_num(hi), f"values between {_rust_num(lo)} and {_rust_num(hi)}")
    @classmethod
    def not_empty(cls, column): return cls._pred(column, "LENGTH({c}) > 0", "non-empty strings")
    @classmethod
    def valid_utf8(cls, column): return cls._pred(column, "{c} IS NOT NULL", "valid UTF-8 strings")
    @classmethod
    def max_bytes(cls, column, n): return cls._pred(column, "OCTET_LENGTH({c}) <= " + str(int(n)), f"strings with max {int(n)} bytes")
    @classmethod
    def past_date(cls, column): return cls._pred(column, "{c} < CURRENT_DATE", "past dates")
    @classmethod
    def future_date(cls, column): return cls._pred(column, "{c} > CURRENT_DATE", "future dates")
    @classmethod
    def date_range(cls, column, start, end): return cls._pred(column, "{c} BETWEEN '" + start + "' AND '" + end + "'", f"dates between {start} and {end}")
    @classmethod
    def valid_timezone(cls, column): return cls._pred(column, "{c} IS NOT NULL", "valid timezone")

    @classmethod
    def custom(cls, column, sql_predicate):
        if ";" in sql_predicate or "drop" in sql_predicate.lower():  # datatype.rs:219-225
            raise ValueError("Potentially unsafe SQL predicate")
        return cls(column, "predicate", sql_predicate.replace("{column}", cls._esc(column)), f"custom validation: {sql_predicate}")

    def _add_to(self, plan):
        # slot = the non-NULL count of the column (also what makes a missing column an error); the predicate count rides behind it
        self._count_slot = None
        s = CompletenessAnalyzer(self.column)._add_to(plan)
        if self.kind == "predicate":
            self._count_slot = ComplianceAnalyzer("datatype", f"{self._esc(self.column)} IS NOT NULL AND ({self.predicate})")._add_to(plan)
        return s

    def _result(self, plan, slot):
        a = plan.analyzer_result(slot)
        if a.error == 2:
            return ConstraintResult(ConstraintStatus.Failure, None, "Error evaluating constraint: " + (a.message or ""), "datatype")
        if self.kind == "specific":
            sch = getattr(plan, "_ctx_schema", None)
            actual = arrow_type_debug(sch.field(self.column).type) if sch is not None else None
            if actual is None:
                return ConstraintResult(ConstraintStatus.Failure, None, "Error evaluating constraint: the table's Arrow schema is not known to this context", "datatype")
            if actual == self.expected:
                return ConstraintResult(ConstraintStatus.Success, 1.0, f"Column '{self.column}' has expected type {self.expected}", "datatype")
            return ConstraintResult(ConstraintStatus.Failure, 0.0, f"Column '{self.column}' has type {actual}, expected {self.expected}", "datatype")
        if self.kind == "consistency":
            consistency = 0.95  # the reference's placeholder (datatype.rs:357-359)
            ok = consistency >= self.threshold
            return ConstraintResult(ConstraintStatus.Success if ok else ConstraintStatus.Failure, consistency,
                                    f"Type consistency {consistency * 100.0:.1f}% {'meets' if ok else 'below'} threshold {self.threshold * 100.0:.1f}%", "datatype")
        c = plan.analyzer_result(self._count_slot)
        if c.error == 2:
            return ConstraintResult(ConstraintStatus.Failure, None, "Error evaluating constraint: " + (c.message or ""), "datatype")
        total, valid = a.u[1], c.u[0]   # CompletenessAnalyzer: u = [rows, non-NULL rows]; ComplianceAnalyzer: u = [satisfied, rows]
        rate = valid / total if total else float("nan")   # SUM over no rows is NULL, read as 0: 0 / 0
        return ConstraintResult(ConstraintStatus.Success if rate >= 1.0 else ConstraintStatus.Failure, rate,
                                f"{_rust_fixed1(rate * 100.0)}% of values satisfy {self.description}", "datatype")


class TemporalOrderingConstraint(Constraint):  # constraints/temporal_ordering.rs:56-600
    """before_after / before_or_equal (with tolerance_seconds), date_range and business_hours (UTC) over the timestamp columns
    of ONE table, as counts of the reference's own comparisons (K1 predicate units): total_rows = the rows its WHERE clause
    keeps, violations = those for which the comparison is not TRUE. The reference's quirk is kept: before_or_equal compares
    with `>` and before_after with `>=` (temporal_ordering.rs:351-367). max_time_gap (LAG window), event sequences and
    business hours in a named time zone are not built: an error result."""
    _UNITS = {"s": 1, "ms": 10**3, "us": 10**6, "ns": 10**9}

    def __init__(self, table_name):
        self.table_name, self.kind, self.args = table_name, "before_after", ("", "", False)
        self._allow_nulls, self._tolerance = False, 0

    def before_after(self, before, after):
        self.kind, self.args = "before_after", (before, after, False)
        return self

    def before_or_equal(self, before, after):
        self.kind, self.args = "before_after", (before, after, True)
        return self

    def business_hours(self, column, start, end):
        self.kind, self.args = "business_hours", [column, start, end, False, None]
        return self

    def weekdays_only(self, flag):
        if self.kind == "business_hours":
            self.args[3] = bool(flag)
        return self

    def with_timezone(self, tz):
        if self.kind == "business_hours":
            self.args[4] = tz
        return self

    def date_range(self, column, min_date=None, max_date=None):
        self.kind, self.args = "date_range", (column, min_date, max_date)
        return self

    def max_time_gap(self, column, max_gap_seconds):
        self.kind, self.args = "max_time_gap", (column, max_gap_seconds)
        return self

    def allow_nulls(self, allow):
        self._allow_nulls = bool(allow)
        return self

    def tolerance_seconds(self, seconds):
        self._tolerance = int(seconds)
        return self

    @staticmethod
    def _q(c): return '"' + c.replace('"', '""') + '"'

    def _unit(self, ctx, column):
        sch = getattr(ctx, "_schemas", {}).get(self.table_name)
        if sch is None or column not in sch.names or not pa.types.is_timestamp(sch.field(column).type):
            raise ValueError(f"'{column}' of table '{self.table_name}' is not a timestamp column known to this context")
        return self._UNITS[sch.field(column).type.unit]

    def _queries(self, ctx):
        """(WHERE clause or None, comparison) — both in the declared predicate grammar"""
        for name in [self.table_name] + (list(self.args[:2]) if self.kind == "before_after" else [self.args[0]]):
            F.check(F.lib().tg_validate_identifier(name.encode()))
        if self.kind == "before_after":
            b, a, allow_equal = self.args
            qb, qa = self._q(b), self._q(a)
            op = ">" if allow_equal else ">="   # (sic: temporal_ordering.rs:351-367)
            rhs = qb
            if self._tolerance > 0:
                ub, ua = self._unit(ctx, b), self._unit(ctx, a)
                if ub != ua:
                    raise ValueError("tolerance_seconds needs both columns in the same timestamp unit")
                rhs = f"{qb} + {self._tolerance * ub}"
            where = None if self._allow_nulls else f"{qb} IS NOT NULL AND {qa} IS NOT NULL"
            return where, f"{qa} {op} {rhs}"
        if self.kind == "date_range":
            c, lo, hi = self.args
            qc = self._q(c)
            conds = ([f"{qc} >= TIMESTAMP '{lo}'"] if lo is not None else []) + ([f"{qc} <= TIMESTAMP '{hi}'"] if hi is not None else [])
            if not conds:
                raise ValueError("DateRange validation requires at least min_date or max_date")
            return (None if self._allow_nulls else f"{qc} IS NOT NULL"), " AND ".join(conds)
        if self.kind == "business_hours":
            c, start, end, weekdays, tz = self.args
            if tz is not None:
                raise ValueError("business hours in a named time zone are not supported (UTC only)")
            u = self._unit(ctx, c)
            qc, day = self._q(c), 86400 * u
            tod = f"((({qc} % {day}) + {day}) % {day})"   # CAST(ts AS TIME) of a naive timestamp, in the column's unit
            sec = lambda hhmm: (int(hhmm.split(":")[0]) * 3600 + int(hhmm.split(":")[1]) * 60) * u
            check = f"{tod} BETWEEN {sec(start)} AND {sec(end)}"
            clauses = []
            if weekdays:  # EXTRACT(DOW ..): Sunday = 0; 1970-01-01 was a Thursday
                clauses.append(f"((((({qc} - {tod}) / {day}) % 7) + 11) % 7) BETWEEN 1 AND 5")
            if not self._allow_nulls:
                clauses.append(f"{qc} IS NOT NULL")
            return (" AND ".join(clauses) if clauses else None), check
        raise ValueError(f"temporal validation '{self.kind}' is not supported (window functions)")

    def _add_to(self, plan):
        return SizeConstraint(Assertion.GreaterThanOrEqual(0.0))._add_to(plan)  # placeholder slot: the constraint names its own table

    def evaluate(self, ctx, table=None):
        try:
            where, cmp_ = self._queries(ctx)
        except (ValueError, F.TermGpuError) as ex:
            return ConstraintResult(ConstraintStatus.Failure, None, f"Error evaluating constraint: {ex}", "temporal_ordering")
        plan = Plan()
        s_ok = ComplianceAnalyzer("ok", f"({where}) AND ({cmp_})" if where else cmp_)._add_to(plan)
        s_tot = ComplianceAnalyzer("total", where)._add_to(plan) if where else None
        plan.execute(ctx, self.table_name)
        ok = plan.analyzer_result(s_ok)
        tot = plan.analyzer_result(s_tot) if s_tot is not None else None
        for a in (ok, tot):
            if a is not None and a.error == 2:
                return ConstraintResult(ConstraintStatus.Failure, None, "Error evaluating constraint: " + (a.message or ""), "temporal_ordering")
        total_rows = tot.u[0] if tot is not None else ok.u[1]
        violations = total_rows - ok.u[0]
        if violations == 0:
            return ConstraintResult(ConstraintStatus.Success, 1.0, None, "temporal_ordering")
        rate = (total_rows - violations) / total_rows if total_rows > 0 else 1.0
        pct = f"{rate * 100.0:.2f}"
        if self.kind == "before_after":
            msg = f"Temporal ordering violation: {violations} records where '{self.args[0]}' is not before '{self.args[1]}' ({pct}% compliance)"
        elif self.kind == "business_hours":
            msg = f"Business hours violation: {violations} records with '{self.args[0]}' outside business hours ({pct}% compliance)"
        else:
            msg = f"Date range violation: {violations} records with '{self.args[0]}' outside valid range ({pct}% compliance)"
        return ConstraintResult(ConstraintStatus.Failure, rate, msg, "temporal_ordering")

    def _result(self, plan, slot):
        ctx = getattr(plan, "_ctx", None)
        if ctx is None:  # (a plan driven through execute_partial / the distributed path by hand: evaluate the constraint directly)
            return ConstraintResult(ConstraintStatus.Failure, None, "Error evaluating constraint: this constraint names its own tables; call evaluate(ctx)", self.__class__.__name__)
        return self.evaluate(ctx)


class CrossTableSumConstraint(Constraint):  # constraints/cross_table_sum.rs:60-630
    """SUM(left_table.col) against SUM(right_table.col) within a tolerance: two K1 sum aggregates, one plan per table, compared on the
    host like the reference's scalar query (:200-215). The grouped form (GROUP BY + FULL OUTER JOIN of per-group sums) is not
    built: an error result. The failure message carries the reference's 'ALL' example row (:296-312, :452-460)."""

    def __init__(self, left_column, right_column):
        self.left_column, self.right_column = left_column, right_column
        self.group_by_columns, self._tolerance, self._max_violations = [], 0.0, 100

    def group_by(self, columns):
        self.group_by_columns = list(columns)
        return self

    def tolerance(self, t):
        self._tolerance = abs(float(t))
        return self

    def max_violations_reported(self, n):
        self._max_violations = int(n)
        return self

    @staticmethod
    def parse_qualified_column(q):
        parts = q.split(".")
        if len(parts) != 2:
            raise ValueError(f"Column must be qualified (table.column): '{q}'")
        for part in parts:
            F.check(F.lib().tg_validate_identifier(part.encode()))
        return parts[0], parts[1]

    @staticmethod
    def _sum(ctx, table, column):
        plan = Plan()
        slot = StatisticalConstraint(column, StatisticType.Sum, Assertion.GreaterThanOrEqual(float("-inf")))._add_to(plan)
        plan.execute(ctx, table)
        r = plan.result(slot)
        if r.error_code:
            raise ValueError(r.message or "sum failed")
        return 0.0 if r.metric is None else float(r.metric)   # COALESCE(SUM(..), 0.0): no non-NULL row

    def _add_to(self, plan):
        return SizeConstraint(Assertion.GreaterThanOrEqual(0.0))._add_to(plan)  # placeholder slot: the constraint names its own tables

    def evaluate(self, ctx, table=None):
        try:
            lt, lc = self.parse_qualified_column(self.left_column)
            rt, rc = self.parse_qualified_column(self.right_column)
            for g in self.group_by_columns:
                F.check(F.lib().tg_validate_identifier(g.encode()))
            if self.group_by_columns:
                raise ValueError("grouped cross-table sums are not supported (per-group sums + FULL OUTER JOIN)")
            left, right = self._sum(ctx, lt, lc), self._sum(ctx, rt, rc)
        except (ValueError, F.TermGpuError) as ex:
            return ConstraintResult(ConstraintStatus.Failure, None, f"Error evaluating constraint: {ex}", "cross_table_sum")
        diff = abs(left - right)
        if not diff > self._tolerance:
            return ConstraintResult(ConstraintStatus.Success, diff, None, "cross_table_sum")
        tol = f" (tolerance: {self._tolerance:.4f})" if self._tolerance > 0.0 else " (exact match required)"
        if self._max_violations > 0:
            ex = f"Group 'ALL': {self.left_column} = {left:.4f}, {self.right_column} = {right:.4f} (diff: {diff:.4f})"
            msg = f"Cross-table sum mismatch: 1/1 overall totals failed validation{tol}. Examples: [{ex}]"
        else:
            msg = (f"Cross-table sum mismatch: 1/1 overall totals failed validation{tol}, total sums: {_rust_num(left)} vs {_rust_num(right)} "
                   f"(max diff: {diff:.4f})")
        return ConstraintResult(ConstraintStatus.Failure, diff, msg, "cross_table_sum")

    def _result(self, plan, slot):
        ctx = getattr(plan, "_ctx", None)
        if ctx is None:  # (a plan driven through execute_partial / the distributed path by hand: evaluate the constraint directly)
            return ConstraintResult(ConstraintStatus.Failure, None, "Error evaluating constraint: this constraint names its own tables; call evaluate(ctx)", self.__class__.__name__)
        return self.evaluate(ctx)


class CoverageType(enum.Enum):  # constraints/join_coverage.rs:72-79
    LeftCoverage = 0
    RightCoverage = 1
    BidirectionalCoverage = 2


class JoinCoverageConstraint(Constraint):  # constraints/join_coverage.rs:61-426
    """Share of the rows of one table whose join key finds a partner in the other: the foreign-key kernels (K3 build / probe) give
    the unmatched rows, the uniqueness kernels verify the precondition under which a LEFT / RIGHT JOIN's row count is the
    table's own — the probed side's keys must be unique (a duplicated key multiplies the join's rows: that needs a counting
    hash join, which is not built: an error result, like composite keys). distinct_only keeps the reference's arithmetic
    (matched ROWS over COUNT(DISTINCT left key)). The count in "(N unmatched examples found)" is the reference's first result
    batch of a DISTINCT .. LIMIT query: here min(distinct unmatched keys, max_examples_reported) — unpinned (it depends on how
    DataFusion partitions the aggregate's output)."""

    def __init__(self, left_table, right_table):
        self.left_table, self.right_table, self.join_keys = left_table, right_table, []
        self.expected_match_rate, self._coverage, self._distinct_only, self._max_examples = 1.0, CoverageType.LeftCoverage, False, 100

    def on(self, left_column, right_column):
        self.join_keys = [(left_column, right_column)]
        return self

    def on_multiple(self, keys):
        self.join_keys = [(l, r) for l, r in keys]
        return self

    def expect_match_rate(self, rate):
        self.expected_match_rate = min(max(float(rate), 0.0), 1.0)
        return self

    def coverage_type(self, t):
        self._coverage = t
        return self

    def distinct_only(self, flag):
        self._distinct_only = bool(flag)
        return self

    def max_examples_reported(self, n):
        self._max_examples = int(n)
        return self

    def _add_to(self, plan):
        return SizeConstraint(Assertion.GreaterThanOrEqual(0.0))._add_to(plan)  # placeholder slot: the constraint names its own tables

    @staticmethod
    def _side(ctx, table, key):
        """(rows, non-NULL keys, distinct keys) of one side"""
        d = DistinctnessAnalyzer(key).compute(ctx, table)
        if d.error == 2:
            raise ValueError(d.message or "join key not readable")
        c = CompletenessAnalyzer(key).compute(ctx, table)
        return c.u[0], c.u[1], d.u[1]

    @staticmethod
    def _unmatched(ctx, child_table, child_key, parent_table, parent_key):
        """(rows of `child` whose non-NULL key has no partner in `parent`, distinct such keys)"""
        r = ForeignKeyConstraint(f"{child_table}.{child_key}", f"{parent_table}.{parent_key}").allow_nulls(True).evaluate(ctx)
        if r.error_code:
            raise ValueError(r.message or "foreign key job failed")
        if r.status is ConstraintStatus.Success:
            return 0, 0
        uniq = int(r.message.split("unique: ")[1].split(")")[0])
        return int(r.metric), uniq

    def evaluate(self, ctx, table=None):
        try:
            for name in [self.left_table, self.right_table] + [c for pair in self.join_keys for c in pair]:
                F.check(F.lib().tg_validate_identifier(name.encode()))
            if not self.join_keys:
                raise ValueError("No join keys specified. Use .on() or .on_multiple() to set join keys")
            if len(self.join_keys) > 1:
                raise ValueError("composite join keys are not supported")
            lk, rk = self.join_keys[0]
            n_l, nn_l, d_l = self._side(ctx, self.left_table, lk)
            n_r, nn_r, d_r = self._side(ctx, self.right_table, rk)
            need_right_unique = self._coverage in (CoverageType.LeftCoverage, CoverageType.BidirectionalCoverage)
            need_left_unique = self._coverage in (CoverageType.RightCoverage, CoverageType.BidirectionalCoverage)
            if (need_right_unique and d_r != nn_r) or (need_left_unique and d_l != nn_l):
                raise ValueError("join coverage over a duplicated key on the probed side is not supported (the join multiplies its rows)")
            if self._distinct_only and self._coverage is not CoverageType.LeftCoverage:
                raise ValueError("distinct_only is supported for LeftCoverage only")
            div = lambda a, b: a / b if b else float("nan")
            examples = 0
            if self._coverage is CoverageType.LeftCoverage:
                orphans, uniq = self._unmatched(ctx, self.left_table, lk, self.right_table, rk)
                matched = nn_l - orphans
                rate = div(matched, d_l if self._distinct_only else n_l)
                examples = uniq + (1 if n_l > nn_l else 0)
            elif self._coverage is CoverageType.RightCoverage:
                orphans, _ = self._unmatched(ctx, self.right_table, rk, self.left_table, lk)
                rate = div(nn_r - orphans, n_r)
            else:
                lo, uniq = self._unmatched(ctx, self.left_table, lk, self.right_table, rk)
                ro, _ = self._unmatched(ctx, self.right_table, rk, self.left_table, lk)
                a, b = div(nn_l - lo, n_l), div(nn_r - ro, n_r)
                rate = float("nan") if (a != a or b != b) else min(a, b)
                examples = uniq + (1 if n_l > nn_l else 0)
            if self._coverage is CoverageType.RightCoverage:  # (the unmatched query is always the LEFT JOIN one: join_coverage.rs:288-324)
                _, uniq = self._unmatched(ctx, self.left_table, lk, self.right_table, rk)
                examples = uniq + (1 if n_l > nn_l else 0)
        except (ValueError, F.TermGpuError) as ex:
            return ConstraintResult(ConstraintStatus.Failure, None, f"Error evaluating constraint: {ex}", "join_coverage")
        if rate >= self.expected_match_rate:
            return ConstraintResult(ConstraintStatus.Success, rate, None, "join_coverage")
        arrow = {CoverageType.LeftCoverage: "->", CoverageType.RightCoverage: "<-", CoverageType.BidirectionalCoverage: "<->"}[self._coverage]
        shown = min(examples, self._max_examples)
        ex_msg = f" ({shown} unmatched examples found)" if self._max_examples > 0 and shown > 0 else ""
        pct = lambda x: "NaN" if x != x else f"{x * 100.0:.2f}"
        return ConstraintResult(ConstraintStatus.Failure, rate,
                                f"Join coverage constraint failed: {self.left_table} {arrow} {self.right_table} coverage is {pct(rate)}% "
                                f"(expected: {pct(self.expected_match_rate)}%){ex_msg}", "join_coverage")

    def _result(self, plan, slot):
        ctx = getattr(plan, "_ctx", None)
        if ctx is None:  # (a plan driven through execute_partial / the distributed path by hand: evaluate the constraint directly)
            return ConstraintResult(ConstraintStatus.Failure, None, "Error evaluating constraint: this constraint names its own tables; call evaluate(ctx)", self.__class__.__name__)
        return self.evaluate(ctx)


def _rust_num(x) -> str:
    """`{}` of an f64 (Range { min, max } are f64 in the reference): integral values print without a fraction"""
    x = float(x)
    return str(int(x)) if x == int(x) and abs(x) < 1e15 else repr(x)


def _rust_fixed1(x: float) -> str:
    return "NaN" if x != x else f"{x:.1f}"


@dataclass
class Check:  # core/check.rs
    name: str
    level: Level = Level.Error
    description: Optional[str] = None
    constraints: List[Constraint] = field(default_factory=list)

    @staticmethod
    def builder(name):
        return CheckBuilder(name)


class CheckBuilder:  # core/check.rs (builder methods listed in SURVEY §0.1)
    def __init__(self, name):
        self._c = Check(name)

    def level(self, lvl: Level):
        self._c.level = lvl
        return self

    def description(self, d):
        self._c.description = d
        return self

    def constraint(self, c: Constraint):
        self._c.constraints.append(c)
        return self

    def has_size(self, assertion): return self.constraint(SizeConstraint(assertion))
    def completeness(self, columns, threshold=1.0, operator=None): return self.constraint(CompletenessConstraint(columns, threshold, operator))
    def validates_uniqueness(self, columns, threshold=1.0): return self.constraint(UniquenessConstraint(columns, UniquenessType.FullUniqueness, threshold))
    def validates_distinctness(self, columns, assertion): return self.constraint(UniquenessConstraint.distinctness(columns, assertion))
    def validates_unique_value_ratio(self, columns, assertion): return self.constraint(UniquenessConstraint.unique_value_ratio(columns, assertion))
    def validates_primary_key(self, columns): return self.constraint(UniquenessConstraint.primary_key(columns))
    def validates_uniqueness_with_nulls(self, columns, threshold, null_handling): return self.constraint(UniquenessConstraint.unique_with_nulls(columns, threshold, null_handling))
    def validates_regex(self, column, pattern, threshold): return self.constraint(FormatConstraint.regex(column, pattern, threshold))
    def validates_email(self, column, threshold): return self.constraint(FormatConstraint.email(column, threshold))
    def validates_url(self, column, threshold, allow_localhost=False): return self.constraint(FormatConstraint.url(column, threshold, allow_localhost))
    def validates_credit_card(self, column, threshold, detect_only): return self.constraint(FormatConstraint.credit_card(column, threshold, detect_only))
    def contains_ssn(self, column, threshold): return self.constraint(FormatConstraint.social_security_number(column, threshold))
    def has_format(self, column, format, threshold, options=None, arg=None, flag=False): return self.constraint(FormatConstraint(column, format, threshold, options, arg, flag))
    def statistic(self, column, stat, assertion, percentile=0.0): return self.constraint(StatisticalConstraint(column, stat, assertion, percentile))
    def has_min(self, column, assertion): return self.statistic(column, StatisticType.Min, assertion)
    def has_max(self, column, assertion): return self.statistic(column, StatisticType.Max, assertion)
    def has_mean(self, column, assertion): return self.statistic(column, StatisticType.Mean, assertion)
    def has_sum(self, column, assertion): return self.statistic(column, StatisticType.Sum, assertion)
    def has_standard_deviation(self, column, assertion): return self.statistic(column, StatisticType.StandardDeviation, assertion)
    def has_variance(self, column, assertion): return self.statistic(column, StatisticType.Variance, assertion)
    def has_correlation(self, c1, c2, assertion): return self.constraint(CorrelationConstraint.pearson(c1, c2, assertion))
    def satisfies(self, expression, hint=None): return self.constraint(CustomSqlConstraint(expression, hint))
    def has_consistent_data_type(self, column, threshold): return self.constraint(UnifiedDataTypeConstraint.type_consistency(column, threshold))  # core/check.rs:651-657
    def cross_table_sum(self, left_column, right_column): return self.constraint(CrossTableSumConstraint(left_column, right_column))  # core/check.rs
    def join_coverage(self, left_table, right_table): return self.constraint(JoinCoverageConstraint(left_table, right_table))  # core/check.rs
    def temporal_ordering(self, table_name): return self.constraint(TemporalOrderingConstraint(table_name))  # core/check.rs:2174-2179
    # core/check.rs has_histogram / has_histogram_with_description
    def has_histogram(self, column, assertion): return self.constraint(HistogramConstraint(column, assertion))
    def has_histogram_with_description(self, column, assertion, description): return self.constraint(HistogramConstraint(column, assertion, description))
    # core/check.rs:518-625, 1777-1786
    def has_column_count(self, assertion): return self.constraint(ColumnCountConstraint(assertion))
    def has_approx_count_distinct(self, column, assertion): return self.constraint(ApproxCountDistinctConstraint(column, assertion))
    def has_min_length(self, column, n): return self.constraint(LengthConstraint.min(column, n))
    def has_max_length(self, column, n): return self.constraint(LengthConstraint.max(column, n))
    def has_length_between(self, column, a, b): return self.constraint(LengthConstraint.between(column, a, b))
    def has_exact_length(self, column, n): return self.constraint(LengthConstraint.exactly(column, n))
    def is_not_empty(self, column): return self.constraint(LengthConstraint.not_empty(column))
    def length(self, column, assertion): return self.constraint(LengthConstraint(column, assertion))
    def foreign_key(self, child, parent): return self.constraint(ForeignKeyConstraint(child, parent))
    # core/check.rs:2233-2298 (completeness with a logical operator over the columns)
    def any_complete(self, columns): return self.completeness(list(columns), 1.0, LogicalOperator.Any)
    def at_least_complete(self, n, columns, threshold): return self.completeness(list(columns), threshold, LogicalOperator.AtLeast(n))
    def exactly_complete(self, n, columns, threshold): return self.completeness(list(columns), threshold, LogicalOperator.Exactly(n))
    # core/check.rs:1019-1222 (format shorthands) and :1259-1410 (the same with FormatOptions)
    def validates_phone(self, column, threshold, country=None): return self.constraint(FormatConstraint.phone(column, threshold, country))
    def validates_postal_code(self, column, threshold, country): return self.constraint(FormatConstraint.postal_code(column, threshold, country))
    def validates_uuid(self, column, threshold): return self.constraint(FormatConstraint.uuid(column, threshold))
    def validates_ipv4(self, column, threshold): return self.constraint(FormatConstraint.ipv4(column, threshold))
    def validates_ipv6(self, column, threshold): return self.constraint(FormatConstraint.ipv6(column, threshold))
    def validates_json(self, column, threshold): return self.constraint(FormatConstraint.json(column, threshold))
    def validates_iso8601_datetime(self, column, threshold): return self.constraint(FormatConstraint.iso8601_datetime(column, threshold))
    def validates_email_with_options(self, column, threshold, options): return self.constraint(FormatConstraint(column, FormatType.Email, threshold, options))
    def validates_url_with_options(self, column, threshold, allow_localhost, options): return self.constraint(FormatConstraint(column, FormatType.Url, threshold, options, flag=allow_localhost))
    def validates_phone_with_options(self, column, threshold, country, options): return self.constraint(FormatConstraint(column, FormatType.Phone, threshold, options, arg=country))
    def validates_regex_with_options(self, column, pattern, threshold, options): return self.constraint(FormatConstraint(column, FormatType.Regex, threshold, options, arg=pattern))
    # core/check.rs:446-457: CorrelationConstraint::mutual_information — the reference answers Skipped (correlation.rs:340-345)
    def has_mutual_information(self, c1, c2, assertion): return self.constraint(CorrelationConstraint(c1, c2, CorrelationType.MutualInformation, assertion))
    # core/check.rs:1480-1500: uniqueness(columns, type, UniquenessOptions{threshold | assertion, null_handling})
    def uniqueness(self, columns, uniqueness_type, threshold=1.0, assertion=None, null_handling=NullHandling.Exclude):
        return self.constraint(UniquenessConstraint(columns, uniqueness_type, threshold, assertion, null_handling))
    def with_constraint(self, c): return self.constraint(c)  # core/check.rs with_constraint
    def constraints(self, cs):
        for c in cs:
            self.constraint(c)
        return self
    def has_approx_quantile(self, column, q, assertion): return self.constraint(QuantileConstraint.percentile(column, q, assertion))  # core/check.rs has_approx_quantile
    def quantile(self, c: 'QuantileConstraint'): return self.constraint(c)

    def build(self) -> Check:
        return self._c


@dataclass
class ValidationIssue:  # core/result.rs:49-70
    check_name: str
    constraint_name: str
    level: Level
    message: str
    metric: Optional[float] = None


@dataclass
class ValidationMetrics:  # core/result.rs:8-46
    total_checks: int = 0
    passed_checks: int = 0
    failed_checks: int = 0
    skipped_checks: int = 0
    execution_time_ms: int = 0
    custom_metrics: Dict[str, float] = field(default_factory=dict)


@dataclass
class ValidationReport:  # core/result.rs:72-118
    suite_name: str
    metrics: ValidationMetrics = field(default_factory=ValidationMetrics)
    issues: List[ValidationIssue] = field(default_factory=list)
    results: List[ConstraintResult] = field(default_factory=list)


@dataclass
class ValidationResult:  # core/result.rs:120-136
    success: bool
    report: ValidationReport

    def is_success(self):
        return self.success

    def is_failure(self):
        return not self.success


class ValidationSuite:  # core/suite.rs
    def __init__(self, name, checks=None, table_name="data"):
        self.name, self.checks, self.table_name = name, list(checks or []), table_name

    @staticmethod
    def builder(name):
        return ValidationSuiteBuilder(name)

    def build_plan(self):
        plan = Plan()
        slots = []
        for check in self.checks:
            for c in check.constraints:
                slots.append((check, c, c._add_to(plan)))
        return plan, slots

    def run(self, ctx: SessionContext, distributed: bool = False) -> ValidationResult:
        """core/suite.rs:399-501 with run_sequential's reporting (:67-258) over ONE fused plan."""
        t0 = time.perf_counter()
        plan, slots = self.build_plan()
        if distributed:
            from .distributed import execute_distributed
            execute_distributed(plan, ctx, self.table_name)
        else:
            plan.execute(ctx, self.table_name)
        report = ValidationReport(self.name)
        m = report.metrics
        has_errors = False
        for check, c, slot in slots:
            r = c._result(plan, slot)
            report.results.append(r)
            m.total_checks += 1
            if r.status is ConstraintStatus.Success:
                m.passed_checks += 1
            elif r.status is ConstraintStatus.Skipped:
                m.skipped_checks += 1
            else:
                m.failed_checks += 1
                if check.level is Level.Error:
                    has_errors = True
                report.issues.append(ValidationIssue(check.name, r.name, check.level,
                                                     r.message or "Constraint failed", r.metric))
            if r.metric is not None:
                m.custom_metrics[f"{check.name}.{r.name}"] = r.metric  # suite.rs:203-209
        m.execution_time_ms = int((time.perf_counter() - t0) * 1000)
        self.last_plan = plan
        return ValidationResult(not has_errors, report)


class ValidationSuiteBuilder:
    def __init__(self, name):
        self._s = ValidationSuite(name)

    def table_name(self, t):
        self._s.table_name = t
        return self

    def check(self, c: Check):
        self._s.checks.append(c)
        return self

    def build(self):
        return self._s


# ----------------------------------------------------------------------------- analyzers ----
class Analyzer:
    """analyzers/traits.rs:65-148: compute_state_from_data + compute_metric_from_state, fused in a plan."""
    KIND = None

    def __init__(self, column=None, column2=None, expression=None):
        self.column, self.column2, self.expression = column, column2, expression

    def _add_to(self, plan):
        return F.check_slot(F.lib().tg_plan_add_analyzer(plan.handle, self.KIND, _opt(self.column),
                                                         _opt(self.column2), _opt(self.expression)))

    def compute(self, ctx, table="data") -> AnalyzerOutput:
        plan = Plan()
        slot = self._add_to(plan)
        plan.execute(ctx, table)
        return plan.analyzer_result(slot)


def _mk(kind, doc):
    return type(doc, (Analyzer,), {"KIND": kind, "__doc__": doc})


class SizeAnalyzer(Analyzer):
    KIND = 0

    def __init__(self):
        super().__init__()


CompletenessAnalyzer = _mk(1, "CompletenessAnalyzer")
DistinctnessAnalyzer = _mk(2, "DistinctnessAnalyzer")
class HistogramAnalyzer(Analyzer):  # analyzers/advanced/histogram.rs
    def __init__(self, column, num_buckets=10):
        super().__init__(column)
        self.num_buckets = num_buckets

    def _add_to(self, plan):
        return F.check_slot(F.lib().tg_plan_add_histogram(plan.handle, self.column.encode(), int(self.num_buckets)))


ApproxCountDistinctAnalyzer = _mk(14, "ApproxCountDistinctAnalyzer")  # advanced/approx_count_distinct.rs (answered exactly)
MeanAnalyzer = _mk(3, "MeanAnalyzer")
MinAnalyzer = _mk(4, "MinAnalyzer")
MaxAnalyzer = _mk(5, "MaxAnalyzer")
SumAnalyzer = _mk(6, "SumAnalyzer")
StandardDeviationAnalyzer = _mk(7, "StandardDeviationAnalyzer")


class CorrelationAnalyzer(Analyzer):
    def __init__(self, c1, c2, kind=8):
        super().__init__(c1, c2)
        self.KIND = kind

    @staticmethod
    def pearson(c1, c2): return CorrelationAnalyzer(c1, c2, 8)
    @staticmethod
    def spearman(c1, c2): return CorrelationAnalyzer(c1, c2, 9)
    @staticmethod
    def covariance(c1, c2): return CorrelationAnalyzer(c1, c2, 10)


class ComplianceAnalyzer(Analyzer):
    KIND = 13

    def __init__(self, name, predicate):
        super().__init__(expression=predicate)
        self.instance = name


class KllSketchAnalyzer(Analyzer):
    def __init__(self, column, k=200, quantiles=(0.25, 0.5, 0.75, 0.9, 0.95, 0.99)):
        super().__init__(column)
        self.k, self.quantiles = k, list(quantiles)

    def _add_to(self, plan):
        q = (C.c_double * max(1, len(self.quantiles)))(*self.quantiles)
        return F.check_slot(F.lib().tg_plan_add_kll(plan.handle, self.column.encode(), self.k, q, len(self.quantiles)))


class GroupedCompletenessAnalyzer(Analyzer):
    """CompletenessAnalyzer::new(c).with_grouping(GroupingConfig::new(cols)) (analyzers/grouped.rs:198-203)"""

    def __init__(self, column, group_columns, max_groups=10000, include_overall=True):
        super().__init__(column)
        self.group_columns, self.max_groups, self.include_overall = list(group_columns), max_groups, include_overall

    def _add_to(self, plan):
        arr, n = _strs(self.group_columns)
        return F.check_slot(F.lib().tg_plan_add_grouped_completeness(plan.handle, self.column.encode(), arr, n,
                                                                     self.max_groups, int(self.include_overall)))


class AnalysisRunner:  # analyzers/runner.rs:149-202 — all analyzers in one plan instead of one scan each
    def __init__(self):
        self.analyzers = []

    def add(self, a: Analyzer):
        self.analyzers.append(a)
        return self

    def run(self, ctx, table="data", distributed=False) -> Dict[str, AnalyzerOutput]:
        plan = Plan()
        slots = [a._add_to(plan) for a in self.analyzers]
        if distributed:
            from .distributed import execute_distributed
            execute_distributed(plan, ctx, table)
        else:
            plan.execute(ctx, table)
        out = {}
        for a, s in zip(self.analyzers, slots):
            r = plan.analyzer_result(s)
            out[r.metric_key] = r
        self.last_plan = plan
        return out
