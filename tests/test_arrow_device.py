"""RecordBatches appended through the Arrow C Device Data Interface (tg_table_append_arrow_device,
SessionContext.register_arrow_device). A CUDA batch is converted in HBM and must leave exactly the state a host append of
the same batch leaves: every buffer record, the meaningful bytes of values, offsets and validity, and a suite's results.
The device arrays are built here from pyarrow buffers copied into torch tensors and exported by the test's own
`__arrow_c_device_array__` (ctypes structs), so every buffer placement, offset and malformed input can be produced."""
import ctypes as C

import numpy as np
import pyarrow as pa
import pytest

import term_b200 as T
from term_b200 import _ffi as F
from tests.test_append_atomic import _state

CPU, CUDA, CUDA_HOST = 1, 2, 3
TG_ERR_INVALID_ARG = 1


# ------------------------------------------------------------------------------- device arrays ----
class ArrowArray(C.Structure):
    pass


ArrowArray._fields_ = [("length", C.c_int64), ("null_count", C.c_int64), ("offset", C.c_int64), ("n_buffers", C.c_int64),
                       ("n_children", C.c_int64), ("buffers", C.POINTER(C.c_void_p)), ("children", C.POINTER(C.POINTER(ArrowArray))),
                       ("dictionary", C.POINTER(ArrowArray)), ("release", C.c_void_p), ("private_data", C.c_void_p)]


class ArrowDeviceArray(C.Structure):
    _fields_ = [("array", ArrowArray), ("device_id", C.c_int64), ("device_type", C.c_int32), ("sync_event", C.c_void_p),
                ("reserved", C.c_int64 * 3)]


assert C.sizeof(ArrowDeviceArray) == 128 and ArrowDeviceArray.device_type.offset == 88 and ArrowDeviceArray.sync_event.offset == 96

_NOOP_RELEASE = C.CFUNCTYPE(None, C.c_void_p)(lambda p: None)  # the engine never calls release; a live array needs one
_capsule_new = C.pythonapi.PyCapsule_New
_capsule_new.restype, _capsule_new.argtypes = C.py_object, [C.c_void_p, C.c_char_p, C.c_void_p]
_SCHEMA, _DEVICE_ARRAY = b"arrow_schema", b"arrow_device_array"


class DeviceBatch:
    """A RecordBatch whose buffers were copied to `place`: "cuda" (torch CUDA tensors), "cuda_host" (pinned torch tensors) or
    "host" (numpy memory, for mislabelling it). With `stream`, the device copies are written on that stream after a delay and
    the batch carries the event recorded behind them."""

    def __init__(self, batch, place="cuda", device_type=None, device_id=0, sizes_on_device=False, stream=None, struct_offset=0):
        import torch
        self.batch, self.place, self.sizes_on_device, self.stream = batch, place, sizes_on_device, stream
        self.keep, self.tensors, self.schemas, self.by_ptr = [], [], [], {}
        if stream is not None:
            stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(stream):
                torch.cuda._sleep(20_000_000)  # the producer is still writing when the call is made
        children = [self._array(col) for col in batch.columns]
        kids = (C.POINTER(ArrowArray) * max(len(children), 1))(*[C.pointer(c) for c in children])
        top = ArrowArray(length=batch.num_rows, null_count=0, offset=struct_offset, n_buffers=1, n_children=len(children),
                         buffers=self._ptrs([0]), children=kids, release=C.cast(_NOOP_RELEASE, C.c_void_p))
        self.keep += [children, kids]
        event = None
        if stream is not None:
            self.event = torch.cuda.Event()
            self.event.record(stream)
            self._ev = C.c_void_p(self.event.cuda_event)
            event = C.addressof(self._ev)
        if device_type is None:
            device_type = {"cuda": CUDA, "cuda_host": CUDA_HOST, "host": CUDA}[place]
        self.dev = ArrowDeviceArray(array=top, device_id=device_id, device_type=device_type, sync_event=event)

    def _ptrs(self, ptrs):
        a = (C.c_void_p * max(len(ptrs), 1))(*ptrs)
        self.keep.append(a)
        return a

    def _place(self, buf, on_device=True):
        import torch
        if buf is None or buf.size == 0:
            return 0
        host = np.frombuffer(buf, dtype=np.uint8).copy()
        if self.place == "host" or not on_device:
            self.keep.append(host)
            return host.ctypes.data
        t = torch.from_numpy(host)
        if self.place == "cuda_host":
            t = t.pin_memory()
        elif self.stream is not None:
            src = t.cuda()
            t = torch.empty_like(src)
            self.stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self.stream):
                t.copy_(src, non_blocking=True)
            self.keep.append(src)
        else:
            t = t.cuda()
        self.tensors.append(t)
        self.by_ptr[t.data_ptr()] = t
        return t.data_ptr()

    def _array(self, arr):
        bufs = list(arr.buffers())
        dictionary = None
        if pa.types.is_dictionary(arr.type):
            bufs = bufs[:2]
            dictionary = C.pointer(self._array(arr.dictionary))
        ptrs = [self._place(b) for b in bufs]
        if arr.type == pa.string_view():
            sizes = pa.py_buffer(np.array([b.size for b in bufs[2:]], dtype=np.int64).tobytes())
            ptrs.append(self._place(sizes, on_device=self.sizes_on_device))
        a = ArrowArray(length=len(arr), null_count=arr.null_count, offset=arr.offset, n_buffers=len(ptrs), n_children=0,
                       buffers=self._ptrs(ptrs), dictionary=dictionary, release=C.cast(_NOOP_RELEASE, C.c_void_p))
        self.keep.append(a)
        return a

    def device_buffer(self, column, k):
        """the tensor holding buffer k of top-level column `column` (to make it malformed after pyarrow validated it)"""
        return self.by_ptr[self.dev.array.children[column].contents.buffers[k]]

    def __arrow_c_device_array__(self, requested_schema=None, **kwargs):
        s = (C.c_uint8 * 72)()
        self.batch.schema._export_to_c(C.addressof(s))
        self.schemas.append(s)
        return _capsule_new(C.addressof(s), _SCHEMA, None), _capsule_new(C.addressof(self.dev), _DEVICE_ARRAY, None)

    def free(self):
        """drops the producer's buffers and overwrites the memory they held"""
        import torch
        n = sum(t.numel() for t in self.tensors if t.is_cuda)
        self.tensors.clear()
        self.by_ptr.clear()
        self.keep.clear()
        junk = torch.full((max(n, 1) * 2,), 0xA5, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        return junk

    def __del__(self):
        for s in self.schemas:  # schemas the engine's caller did not import
            rel = C.cast(C.addressof(s) + 56, C.POINTER(C.c_void_p))[0]
            if rel:
                C.CFUNCTYPE(None, C.c_void_p)(rel)(C.addressof(s))


def _append_dev(tab, obj):
    """one raw tg_table_append_arrow_device call; returns the status"""
    from term_b200.api import _capsule_pointer
    sc, ac = obj.__arrow_c_device_array__()
    return F.lib().tg_table_append_arrow_device(tab, _capsule_pointer(sc, b"arrow_schema"), _capsule_pointer(ac, b"arrow_device_array"))


# ----------------------------------------------------------------------------------------- data ----
TEMPORAL = {"tdD": pa.date32(), "tdm": pa.date64(), "tts": pa.time32("s"), "ttm": pa.time32("ms"), "ttu": pa.time64("us"),
            "ttn": pa.time64("ns"), "tss": pa.timestamp("s"), "tsm": pa.timestamp("ms"), "tsu": pa.timestamp("us", tz="UTC"),
            "tsn": pa.timestamp("ns"), "tDs": pa.duration("s"), "tDm": pa.duration("ms"), "tDu": pa.duration("us"), "tDn": pa.duration("ns")}
INTS = {"l": (pa.int64(), -10**15, 10**15), "i": (pa.int32(), -2**31, 2**31 - 1), "c": (pa.int8(), -128, 127), "C": (pa.uint8(), 0, 255),
        "s": (pa.int16(), -2**15, 2**15 - 1), "S": (pa.uint16(), 0, 2**16 - 1), "I": (pa.uint32(), 0, 2**32 - 1), "L": (pa.uint64(), 0, 2**63 - 1)}
INDEX = {"c": pa.int8(), "C": pa.uint8(), "s": pa.int16(), "S": pa.uint16(), "i": pa.int32(), "I": pa.uint32(), "l": pa.int64(), "L": pa.uint64()}
WORDS = ["", "a", "héllo", "日本語", "x" * 12, "y" * 13, "user@example.com", "long " * 30, "123-45-6789", "z"]
FORMATS = (list(INTS) + ["g", "f", "b", "u", "U", "vu"] + list(TEMPORAL) + [f"dict:{k}:u" for k in INDEX] + [f"dict:{k}:U" for k in INDEX]
           + ["dict:i:u:null"])


def _array(fmt, n, null_p, rng):
    mask = rng.random(n) < null_p if null_p else None
    if null_p == 1.0:
        mask = np.ones(n, dtype=bool)
    if fmt in INTS:
        typ, lo, hi = INTS[fmt]
        return pa.array(rng.integers(lo, hi, n, endpoint=True, dtype=np.int64 if fmt != "L" else np.uint64), type=typ, mask=mask)
    if fmt in ("g", "f"):
        v = rng.normal(50.0, 20.0, n)
        v[rng.random(n) < 0.01] = np.inf
        return pa.array(v.astype(np.float64 if fmt == "g" else np.float32), mask=mask)
    if fmt == "b":
        return pa.array(rng.random(n) < 0.5, mask=mask)
    if fmt in TEMPORAL:
        typ = TEMPORAL[fmt]
        w = 4 if typ in (pa.date32(), pa.time32("s"), pa.time32("ms")) else 8
        hi = 86_399 if fmt in ("tts",) else 86_399_999 if fmt == "ttm" else 10**6 if w == 4 else 10**12
        return pa.array(rng.integers(0, hi, n), mask=mask).cast(pa.int32() if w == 4 else pa.int64()).view(typ)
    words = [WORDS[k] for k in rng.integers(0, len(WORDS), n)]
    if fmt in ("u", "U", "vu"):
        return pa.array(words, type={"u": pa.string(), "U": pa.large_string(), "vu": pa.string_view()}[fmt], mask=mask)
    _, k, vt = fmt.split(":")[:3]
    dict_vals = pa.array(WORDS + (["never"] if k in "cC" else []), type=pa.string() if vt == "u" else pa.large_string(),
                         mask=np.array([i == 3 for i in range(len(WORDS))]) if fmt.endswith(":null") else None)
    codes = rng.integers(0, len(WORDS), n)
    return pa.DictionaryArray.from_arrays(pa.array(codes, type=INDEX[k], mask=mask), dict_vals)


def _batch(fmt, n, null_p, offset, seed, name="x"):
    rng = np.random.default_rng(seed)
    return pa.record_batch([_array(fmt, n + offset, null_p, rng).slice(offset)], names=[name])


def _bytes(ctx, table, column):
    """the meaningful bytes of a column: values, offsets, validity (last partial byte masked)"""
    import torch
    from term_b200.distributed import _tensor_from_ptr
    b = ctx.column_buffers(table, column)
    n, dev = b["n_rows"], torch.device("cuda", 0)

    def read(ptr, k):
        return _tensor_from_ptr(ptr, max(k, 1), dev, "|u1").cpu().numpy()[:k].copy() if ptr else None

    def masked(ptr, bits):
        a = read(ptr, (bits + 7) // 8)
        if a is not None and bits % 8:
            a[-1] &= (1 << (bits % 8)) - 1
        return a

    if b["dtype"] == F.TG_BOOL:
        vals = masked(b["values"], n)
    else:
        vals = read(b["values"], b["n_value_bytes"])
    offs = read(b["offsets"], (n + 1) * 4) if b["dtype"] == F.TG_UTF8 else None
    return vals, offs, masked(b["validity"], n)


def _assert_same_columns(ctx, a, b):
    sa, sb = _state(ctx, a), _state(ctx, b)
    assert sa == sb
    for col in sa[1]:
        for x, y in zip(_bytes(ctx, a, col), _bytes(ctx, b, col)):
            assert (x is None) == (y is None), col
            if x is not None:
                assert x.tobytes() == y.tobytes(), col


NUMERIC = set(INTS) | {"g", "f"}


def _suite(ctx, name, columns):
    """a suite's results over the table; numeric analyzers on numeric columns, lengths on strings, completeness on all"""
    A = T.Assertion
    cb = T.Check.builder("c").has_size(A.GreaterThan(0.0)).has_column_count(A.GreaterThan(0.0))
    for col, fmt in columns.items():
        cb = cb.completeness(col, 0.5)
        if fmt in NUMERIC:
            cb = cb.has_min(col, A.LessThan(1e30)).has_max(col, A.GreaterThan(-1e30)).has_mean(col, A.Between(-1e30, 1e30)).has_sum(col, A.Between(-1e40, 1e40))
        elif fmt in ("u", "U", "vu") or fmt.startswith("dict"):
            cb = cb.has_min_length(col, 0).has_max_length(col, 10**6)
    res = T.ValidationSuite.builder("s").table_name(name).check(cb.build()).build().run(ctx).report.results
    return [repr((r.name, r.status, r.metric, r.message)) for r in res]


def _check_same(ctx, dev_name, host_name, columns):
    _assert_same_columns(ctx, dev_name, host_name)
    assert _suite(ctx, dev_name, columns) == _suite(ctx, host_name, columns)


# ------------------------------------------------------------------------------------------ GPU ----
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FORMATS)
def test_every_format_matches_the_host_append(ctx, fmt):
    """each format, NULL fraction 0 / 5 / 100 %, slice offset 0 / 3 / 13, prime-sized batches"""
    for null_p in (0.0, 0.05, 1.0):
        for offset, n in ((0, 1009), (3, 523), (13, 2053)):
            batch = _batch(fmt, n, null_p, offset, seed=n + offset)
            ctx.register_arrow_device("dev", DeviceBatch(batch))
            ctx.register_table("host", batch)
            try:
                _check_same(ctx, "dev", "host", {"x": fmt})
            finally:
                ctx.deregister_table("dev")
                ctx.deregister_table("host")


@pytest.mark.gpu
def test_int8_min_keeps_the_delivered_type(ctx):
    """MIN over an Int8 column is typed Int8 by DataFusion: the error result shows the device path recorded src_type"""
    batch = _batch("c", 1009, 0.05, 3, seed=1)
    ctx.register_arrow_device("dev", DeviceBatch(batch))
    ctx.register_table("host", batch)
    try:
        got, want = _suite(ctx, "dev", {"x": "c"}), _suite(ctx, "host", {"x": "c"})
        assert got == want
        assert ctx._schemas["dev"] == batch.schema
    finally:
        ctx.deregister_table("dev")
        ctx.deregister_table("host")


INTERLEAVED = ["l", "g", "i", "b", "c", "I", "L", "u", "U", "vu", "tsu", "dict:s:u", "dict:i:u:null"]


@pytest.mark.gpu
def test_interleaved_host_and_device_appends(ctx):
    """host and device appends alternate at unaligned row counts (the first batches without NULLs, so bitmaps are
    materialised late); the table equals one host registration of the concatenation"""
    sizes = [7, 13, 61, 1000, 3, 129, 64, 1, 517]
    batches = []
    for k, n in enumerate(sizes):
        cols = [_batch(f, n, 0.0 if k < 3 else 0.1, k % 5, seed=100 * k + j).column(0) for j, f in enumerate(INTERLEAVED)]
        batches.append(pa.record_batch(cols, names=[f"c{j}" for j in range(len(INTERLEAVED))]))
    tab = ctx._create("dev")
    try:
        for k, b in enumerate(batches):
            if k % 2:
                ctx._append_batch_c(tab, b)
            else:
                F.check(_append_dev(tab, DeviceBatch(b)))
        whole = pa.Table.from_batches([pa.record_batch([pa.concat_arrays([b.column(j) for b in batches]) for j in range(len(INTERLEAVED))],
                                                       names=batches[0].schema.names)])
        ctx.register_table("host", whole)
        _check_same(ctx, "dev", "host", {f"c{j}": f for j, f in enumerate(INTERLEAVED)})
        # one more unaligned append each, after the tail mirrors of both paths
        extra = pa.record_batch([_batch(f, 11, 0.3, 5, seed=7 + j).column(0) for j, f in enumerate(INTERLEAVED)], names=batches[0].schema.names)
        F.check(_append_dev(tab, DeviceBatch(extra)))
        ctx._append_batch_c(_table(ctx, "host"), extra)
        _check_same(ctx, "dev", "host", {f"c{j}": f for j, f in enumerate(INTERLEAVED)})
    finally:
        ctx.deregister_table("dev")
        ctx.deregister_table("host")


def _table(ctx, name):
    t = C.c_void_p()
    F.check(F.lib().tg_table_lookup(ctx.handle, name.encode(), C.byref(t)))
    return t


@pytest.mark.gpu
def test_other_device_types(ctx):
    """pyarrow's own CPU capsule, a CUDA_HOST batch in pinned memory and Utf8View sizes in device memory give the state of
    register_table"""
    cols = ["l", "g", "b", "u", "vu", "dict:C:U", "S"]
    batch = pa.record_batch([_batch(f, 2003, 0.05, 5, seed=j).column(0) for j, f in enumerate(cols)], names=[f"c{j}" for j in range(len(cols))])
    columns = {f"c{j}": f for j, f in enumerate(cols)}
    ctx.register_table("host", batch)
    try:
        for obj in (batch, DeviceBatch(batch, place="cuda_host"), DeviceBatch(batch, sizes_on_device=True)):
            ctx.register_arrow_device("dev", obj)
            try:
                _check_same(ctx, "dev", "host", columns)
            finally:
                ctx.deregister_table("dev")
    finally:
        ctx.deregister_table("host")


@pytest.mark.gpu
def test_sync_event_and_producer_reuse(ctx):
    """a batch written on a side stream is passed with its event; its buffers are freed and overwritten right after the call"""
    import torch
    cols = ["l", "g", "b", "u", "vu", "dict:i:u:null", "c"]
    batches = [pa.record_batch([_batch(f, n, 0.05, 3, seed=n + j).column(0) for j, f in enumerate(cols)], names=[f"c{j}" for j in range(len(cols))])
               for n in (100_003, 70_001)]
    columns = {f"c{j}": f for j, f in enumerate(cols)}
    side = torch.cuda.Stream()
    producers = [DeviceBatch(b, stream=side) for b in batches]
    ctx.register_arrow_device("dev", producers)
    junk = [p.free() for p in producers]
    ctx.register_table("host", batches)
    try:
        _check_same(ctx, "dev", "host", columns)
    finally:
        del junk
        ctx.deregister_table("dev")
        ctx.deregister_table("host")


def _views(n_bytes_data, view_off, length):
    """a 2-row Utf8View array whose second view points at [view_off, view_off + length) of a data buffer of n_bytes_data"""
    views = np.zeros(2, dtype=[("len", "<i4"), ("prefix", "S4"), ("buf", "<i4"), ("off", "<i4")])
    views[0] = (1, b"a", 0, 0)
    views[1] = (length, b"abcd", 0, view_off)
    return pa.Array.from_buffers(pa.string_view(), 2, [None, pa.py_buffer(views.tobytes()), pa.py_buffer(b"a" * n_bytes_data)])


REFUSALS = {
    "uint64_top_bit": (lambda: pa.record_batch([pa.array(np.arange(777, dtype=np.int64)), pa.array(np.where(np.arange(777) == 400, 2**63 + 5, 5).astype(np.uint64))],
                                               names=["a", "u"]), {}, F.TG_ERR_UNSUPPORTED, "above the Int64 range"),
    "dict_index_outside": (lambda: pa.record_batch([pa.array(np.arange(5, dtype=np.int64)),
                                                    pa.DictionaryArray.from_arrays(pa.array([0, 1, 9, 2, 0], type=pa.int32()), pa.array(["p", "q", "r"]), safe=False)],
                                                   names=["a", "d"]), {}, TG_ERR_INVALID_ARG, "outside the dictionary"),
    "dict_index_outside_null_value": (lambda: pa.record_batch([pa.array(np.arange(5, dtype=np.int64)),
                                                               pa.DictionaryArray.from_arrays(pa.array([0, 1, 9, 2, 0], type=pa.int16()),
                                                                                              pa.array(["p", None, "r"]), safe=False)],
                                                              names=["a", "d"]), {}, TG_ERR_INVALID_ARG, "outside the dictionary"),
    "view_outside_buffer": (lambda: pa.record_batch([pa.array([1, 2], type=pa.int64()), _views(40, 30, 20)], names=["a", "v"]), {},
                            TG_ERR_INVALID_ARG, "outside its data buffer"),
    "large_utf8_2gib": (lambda: pa.record_batch([pa.array([1, 2], type=pa.int64()), pa.array(["abcd", "efgh"], type=pa.large_string())], names=["a", "s"]),
                        {}, F.TG_ERR_UNSUPPORTED, "2 GiB"),  # (the last offset is raised past 2 GiB on the device below)
    "wrong_device_id": (lambda: pa.record_batch([pa.array([1, 2], type=pa.int64())], names=["a"]), {"device_id": 5}, TG_ERR_INVALID_ARG, "device 5"),
    "unknown_device_type": (lambda: pa.record_batch([pa.array([1, 2], type=pa.int64())], names=["a"]), {"device_type": 7}, F.TG_ERR_UNSUPPORTED, "device type 7"),
    "host_pointer_as_cuda": (lambda: pa.record_batch([pa.array([1, 2], type=pa.int64()), pa.array(["a", "b"])], names=["a", "s"]), {"place": "host"},
                             TG_ERR_INVALID_ARG, "not device memory"),
    "sliced_struct": (lambda: pa.record_batch([pa.array([1, 2], type=pa.int64())], names=["a"]), {"struct_offset": 1}, F.TG_ERR_UNSUPPORTED, "sliced struct"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(REFUSALS))
def test_refusals_leave_the_table_unchanged(ctx, case):
    import torch
    make, kw, code, text = REFUSALS[case]
    rng = np.random.default_rng(5)
    good = pa.record_batch([pa.array(rng.integers(-100, 100, 1001), mask=rng.random(1001) < 0.1)], names=["a"])
    ctx.register_arrow_device("refuse", DeviceBatch(good))
    try:
        tab = _table(ctx, "refuse")
        before = _state(ctx, "refuse")
        bytes_before = _bytes(ctx, "refuse", "a")
        bad = DeviceBatch(make(), **kw)
        if case == "large_utf8_2gib":  # offsets [0, 4, 2^31 + 4] over 8 bytes of data: refused before the bytes are read
            bad.device_buffer(1, 1).view(torch.int64)[2] = 2**31 + 4
        st = _append_dev(tab, bad)
        assert st == code, F.last_error()
        assert text in F.last_error()
        assert _state(ctx, "refuse") == before
        assert all((x is None and y is None) or x.tobytes() == y.tobytes() for x, y in zip(_bytes(ctx, "refuse", "a"), bytes_before))
        # the table still takes valid data
        F.check(_append_dev(tab, DeviceBatch(good)))
        assert _state(ctx, "refuse")[0] == 2002
    finally:
        ctx.deregister_table("refuse")


@pytest.mark.gpu
def test_at_size(ctx):
    """100 M-row Int64 / Float64 and 25 M-row Utf8 device registrations equal the host registration, compared on the device"""
    import torch
    from term_b200.distributed import _tensor_from_ptr
    rng = np.random.default_rng(9)
    n, ns = 100_000_000, 25_000_000
    lens = rng.integers(0, 24, ns).astype(np.int32)
    offs = np.zeros(ns + 1, dtype=np.int32)
    np.cumsum(lens, out=offs[1:])
    data = rng.integers(97, 123, int(offs[-1]), dtype=np.uint8)
    valid_s = rng.random(ns) >= 0.05
    strings = pa.Array.from_buffers(pa.string(), ns, [pa.array(valid_s).buffers()[1], pa.py_buffer(offs.tobytes()), pa.py_buffer(data.tobytes())],
                                    null_count=int((~valid_s).sum()))
    cases = [pa.record_batch([pa.array(rng.integers(-10**12, 10**12, n), mask=rng.random(n) < 0.05),
                              pa.array(rng.normal(0.0, 1.0, n))], names=["i", "f"]),
             pa.record_batch([strings], names=["s"])]
    dev = torch.device("cuda", 0)
    for batch in cases:
        ctx.register_arrow_device("big_dev", DeviceBatch(batch))
        ctx.register_table("big_host", batch)
        try:
            assert _state(ctx, "big_dev") == _state(ctx, "big_host")
            for col in batch.schema.names:
                a, b = ctx.column_buffers("big_dev", col), ctx.column_buffers("big_host", col)
                rows = a["n_rows"]
                spans = [("values", a["n_value_bytes"]), ("offsets", (rows + 1) * 4 if a["dtype"] == F.TG_UTF8 else 0), ("validity", rows // 8)]
                for key, k in spans:
                    if k:
                        assert bool(a[key]) == bool(b[key])
                        if a[key]:
                            assert torch.equal(_tensor_from_ptr(a[key], k, dev, "|u1"), _tensor_from_ptr(b[key], k, dev, "|u1")), (col, key)
        finally:
            ctx.deregister_table("big_dev")
            ctx.deregister_table("big_host")
