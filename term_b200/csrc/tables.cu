// Arrow buffer marshalling: values, validity bitmaps and Utf8 offsets staged into HBM.
// Replaces MemTable registration on a SessionContext (e.g. constraints/completeness.rs:389-391 in the
// reference tests, sources/mod.rs:48-66 in production) for the GPU path.
#include <algorithm>
#include <cstddef>
#include <cstring>

#include "engine.hpp"
#include "str_entries.cuh"

namespace tg {

static size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Pivot K of the shifted moment sums: the median of the first (up to) five finite, valid values of the
// column. It must be an ELEMENT of the column (the scan replaces NULL rows by K), and a typical one, so
// that sum(x) = n*K + sum(x-K) keeps full accuracy; a median of five is robust to isolated outliers.
void set_pivot_host(Column& c, int32_t dtype, int64_t n, const void* values, const uint8_t* validity,
                    int64_t bit_offset) {
    if (c.pivot_set || (dtype != TG_INT64 && dtype != TG_FLOAT64)) return;
    double cand[5];
    int64_t icand[5];
    int m = 0;
    for (int64_t i = 0; i < n && i < 65536 && m < 5; ++i) {
        bool ok = !validity || ((validity[(bit_offset + i) >> 3] >> ((bit_offset + i) & 7)) & 1);
        if (!ok) continue;
        if (dtype == TG_INT64) {
            icand[m] = reinterpret_cast<const int64_t*>(values)[i];
            cand[m] = (double)icand[m];
            ++m;
        } else {
            double v = reinterpret_cast<const double*>(values)[i];
            if (v == v && v - v == 0.0) {
                cand[m] = v;
                icand[m] = 0;
                ++m;
            }
        }
    }
    if (m == 0) return;
    for (int i = 1; i < m; ++i)
        for (int j = i; j > 0 && (dtype == TG_INT64 ? icand[j] < icand[j - 1] : cand[j] < cand[j - 1]); --j) {
            std::swap(cand[j], cand[j - 1]);
            std::swap(icand[j], icand[j - 1]);
        }
    c.pivot = cand[m / 2];
    c.ipivot = icand[m / 2];
    c.pivot_set = true;
}

// append `n` bits taken from src starting at bit `src_off` (or all-ones when src == nullptr) to a device
// bitmap that currently holds `have` bits; tail = host mirror of its last partial byte
static void append_bits(Engine& e, DevBuf& buf, uint8_t& tail, int64_t have, const uint8_t* src, int64_t src_off,
                        int64_t n, int64_t* zeros) {
    const int64_t total = have + n;
    e.dev_reserve(buf, (size_t)(total + 7) / 8, (size_t)(have + 7) / 8);
    const int64_t first_byte = have / 8;
    const int shift = (int)(have % 8);
    const size_t out_bytes = (size_t)((total + 7) / 8 - first_byte);
    std::vector<uint8_t> tmp(out_bytes + 8, 0);
    if (shift) tmp[0] = tail & (uint8_t)((1u << shift) - 1);
    int64_t z = 0;
    if (!src) {
        for (int64_t i = 0; i < n; ++i) {
            const int64_t o = shift + i;
            tmp[o >> 3] |= (uint8_t)(1u << (o & 7));
        }
    } else if (shift == 0 && (src_off & 7) == 0) {
        memcpy(tmp.data(), src + src_off / 8, (size_t)(n + 7) / 8);
        if (n & 7) tmp[(n - 1) / 8] &= (uint8_t)((1u << (n & 7)) - 1);
        for (size_t i = 0; i < (size_t)(n + 7) / 8; ++i) z += 8 - __builtin_popcount(tmp[i]);
        z -= (8 - (n & 7)) & 7;
    } else {
        for (int64_t i = 0; i < n; ++i) {
            const int64_t s = src_off + i;
            const int bit = (src[s >> 3] >> (s & 7)) & 1;
            const int64_t o = shift + i;
            tmp[o >> 3] |= (uint8_t)(bit << (o & 7));
            z += !bit;
        }
    }
    if (zeros) *zeros = z;
    tail = (total & 7) ? tmp[out_bytes - 1] : 0;
    // staged copy (tmp is pageable; h2d copies it into the pinned ring before returning)
    e.h2d(buf.p + first_byte, tmp.data(), out_bytes);
}

Column* table_get_or_add(Table& t, const std::string& name, int32_t dtype) {
    Column* c = t.find(name);
    if (c) {
        if (c->dtype != dtype) throw Error(TG_ERR_TYPE_MISMATCH, "column '" + name + "' was registered with a different type");
        return c;
    }
    validate_identifier(name);
    auto nc = std::make_unique<Column>();
    nc->name = name;
    nc->dtype = dtype;
    t.cols.push_back(std::move(nc));
    return t.cols.back().get();
}

AppendTxn::AppendTxn(Table& t_) : e(*t_.eng), t(t_), g(e.mu), n_cols(t.cols.size()), n_rows(t.n_rows) {
    TG_CUDA(cudaSetDevice(e.device));
}

Column& AppendTxn::column(const std::string& name, int32_t dtype) {
    Column& c = *table_get_or_add(t, name, dtype);
    if (c.adopted) throw Error(TG_ERR_INVALID_ARG, "cannot append to an adopted device column");
    for (const Saved& s : saved)
        if (s.c == &c) return c;
    saved.push_back(Saved{&c, c.n_rows, c.value_bytes, c.null_count, c.last_offset, c.tail_byte, c.tail_vbyte, c.pivot_set, c.validity.p != nullptr,
                          c.pivot, c.ipivot, c.src_type, c.src_unsigned, c.temporal, c.temporal_unit});
    return c;
}

void AppendTxn::commit() {
    for (const Saved& s : saved) t.n_rows = std::max(t.n_rows, s.c->n_rows);
    committed = true;
}

AppendTxn::~AppendTxn() {
    if (committed) return;
    // copies and kernels of the call may still be writing the buffers freed below
    cudaStreamSynchronize(e.copy_stream);
    if (e.side[0]) cudaStreamSynchronize(e.side[0]);
    for (const Saved& s : saved) {
        Column& c = *s.c;
        c.n_rows = s.n_rows;
        c.value_bytes = s.value_bytes;
        c.null_count = s.null_count;
        c.last_offset = s.last_offset;
        c.tail_byte = s.tail_byte;
        c.tail_vbyte = s.tail_vbyte;
        c.pivot_set = s.pivot_set;
        c.pivot = s.pivot;
        c.ipivot = s.ipivot;
        c.src_type = s.src_type;
        c.src_unsigned = s.src_unsigned;
        c.temporal = s.temporal;
        c.temporal_unit = s.temporal_unit;
        if (!s.had_validity && c.validity.p) {
            if (c.validity.owned) e.dev_free(c.validity.p, c.validity.cap);
            c.validity = DevBuf{};
        }
    }
    while (t.cols.size() > n_cols) {
        column_free(e, *t.cols.back());
        t.cols.pop_back();
    }
    t.n_rows = n_rows;
}

// appends the validity of `n` rows (bitmap `validity` read from bit `bit_offset`; nullptr = no NULLs) to a column that
// holds `have` rows; materialises the bitmap lazily the first time a NULL shows up
void append_validity(Engine& e, Column& c, int64_t have, const uint8_t* validity, int64_t bit_offset, int64_t n) {
    bool has_nulls = false;
    bool fast_bits = false;
    int64_t zeros = 0;
    if (validity) {
        if ((bit_offset & 7) == 0 && (have & 7) == 0) {
            // byte-aligned on both sides: count zero bits 64 at a time; the bitmap bytes then go to the device as
            // they are (direct DMA when the source is pinned)
            const uint8_t* src = validity + bit_offset / 8;
            const int64_t full_words = n / 64;
            int64_t ones = 0;
            for (int64_t w = 0; w < full_words; ++w) {
                uint64_t x;
                memcpy(&x, src + 8 * w, 8);
                ones += __builtin_popcountll(x);
            }
            for (int64_t i = full_words * 64; i < n; ++i) ones += (src[i >> 3] >> (i & 7)) & 1;
            zeros = n - ones;
            has_nulls = zeros > 0;
            fast_bits = true;
        } else {
            for (int64_t i = 0; i < n && !has_nulls; ++i) {
                const int64_t s = bit_offset + i;
                has_nulls = !((validity[s >> 3] >> (s & 7)) & 1);
            }
        }
    }
    if (has_nulls && !c.validity.p && have > 0) {
        // earlier batches had no bitmap: materialise all-ones for them
        append_bits(e, c.validity, c.tail_byte, 0, nullptr, 0, have, nullptr);
    }
    if (has_nulls || c.validity.p) {
        if (fast_bits && validity) {
            const size_t nbytes = (size_t)(n + 7) / 8;
            e.dev_reserve(c.validity, (size_t)(have + n + 7) / 8, (size_t)(have + 7) / 8);
            e.h2d(c.validity.p + have / 8, validity + bit_offset / 8, nbytes);
            // host mirror of the last partial byte (bits past the end masked off) for the next unaligned append
            c.tail_byte = (n & 7) ? (uint8_t)(validity[bit_offset / 8 + nbytes - 1] & ((1u << (n & 7)) - 1)) : 0;
        } else {
            append_bits(e, c.validity, c.tail_byte, have, validity, bit_offset, n, &zeros);
        }
        c.null_count += zeros;
    }
}

// ORs a chunk-relative bitmap (32-bit words) into a column bitmap at bit `have`; the destination bits from `have` on are 0
__global__ void merge_bits_kernel(uint32_t* __restrict__ dst, uint64_t have, const uint32_t* __restrict__ words, uint64_t n_words) {
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t v = words[w];
        if (!v) continue;
        const uint64_t pos = have + 32 * w;
        const uint32_t sh = (uint32_t)(pos & 31);
        atomicOr(dst + (pos >> 5), v << sh);
        if (sh && (v >> (32 - sh))) atomicOr(dst + (pos >> 5) + 1, v >> (32 - sh));
    }
}

// the device counterpart of append_bits: appends n bits of a chunk-relative device bitmap to `buf` (holding `have` bits);
// `tail` (host mirror of the last partial byte) continues from the read-back of the chunk's last 64 bits
void append_bits_device(Engine& e, DevBuf& buf, uint8_t& tail, int64_t have, const uint32_t* words, int64_t n, uint64_t last64) {
    if (n <= 0) return;
    const int64_t total = have + n;
    e.dev_reserve(buf, (size_t)(total + 7) / 8, (size_t)(have + 7) / 8);
    // the partial byte keeps only its earlier rows (a device byte may hold stale bits past them), the bytes after it start at 0
    const uint8_t part = (have & 7) ? (uint8_t)(tail & ((1u << (have & 7)) - 1u)) : 0;
    const size_t b0 = (size_t)have / 8, b1 = (size_t)(total + 7) / 8;
    TG_CUDA(cudaMemsetAsync(buf.p + b0, 0, b1 - b0, e.copy_stream));
    if (part) e.h2d(buf.p + b0, &part, 1);
    const uint64_t n_words = (uint64_t)(n + 31) / 32;
    const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>((n_words + 255) / 256, (uint64_t)e.sm_count * 8));
    merge_bits_kernel<<<grid, 256, 0, e.copy_stream>>>(reinterpret_cast<uint32_t*>(buf.p), (uint64_t)have, words, n_words);
    TG_CUDA(cudaGetLastError());
    e.launches += 1;
    uint8_t t = 0;
    for (int64_t row = total & ~(int64_t)7; row < total; ++row) {
        const int bit = row < have ? (tail >> (row & 7)) & 1 : (int)((last64 >> (row - have - n + 64)) & 1);
        t |= (uint8_t)(bit << (row & 7));
    }
    tail = t;
}

// the device counterpart of append_validity: the bitmap is materialised (all-ones for the earlier rows) when the column
// first sees a NULL, as there
void append_validity_device(Engine& e, Column& c, int64_t have, const uint32_t* words, int64_t n, int64_t zeros, uint64_t last64) {
    if (zeros > 0 && !c.validity.p && have > 0) append_bits(e, c.validity, c.tail_byte, 0, nullptr, 0, have, nullptr);
    if (zeros > 0 || c.validity.p) {
        append_bits_device(e, c.validity, c.tail_byte, have, words, n, last64);
        c.null_count += zeros;
    }
}

// table_append_host inside a caller's transaction (table_append_arrow appends every child of a batch in one)
static void append_host_column(AppendTxn& txn, const std::string& name, int32_t dtype, int64_t n, const void* values,
                               const int32_t* offsets, const uint8_t* validity, int64_t bit_offset) {
    Engine& e = txn.e;
    if (n < 0) throw Error(TG_ERR_INVALID_ARG, "negative row count");
    Column& c = txn.column(name, dtype);
    const int64_t have = c.n_rows;
    if (n == 0) return;
    // ---- fixed-width values first: their DMA (the bulk of the bytes) is queued before the host walks the validity
    // bitmap below, so counting NULLs overlaps the copy instead of delaying it ----
    const bool fixed_width = dtype == TG_INT64 || dtype == TG_FLOAT64 || dtype == TG_INT32 || dtype == TG_FLOAT32;
    if (fixed_width) {
        const size_t w = (size_t)c.elem_bytes();
        e.dev_reserve(c.values, (size_t)(have + n) * w, (size_t)have * w);
        e.h2d(c.values.p + (size_t)have * w, values, (size_t)n * w);
        c.value_bytes = (have + n) * (int64_t)w;
        set_pivot_host(c, dtype, n, values, validity, bit_offset);
    }
    append_validity(e, c, have, validity, bit_offset, n);
    // ---- values ----
    switch (dtype) {
        case TG_INT64:
        case TG_FLOAT64:
        case TG_INT32:
        case TG_FLOAT32: break;  // queued above
        case TG_BOOL: {
            append_bits(e, c.values, c.tail_vbyte, have, (const uint8_t*)values, bit_offset, n, nullptr);
            c.value_bytes = (have + n + 7) / 8;
        } break;
        case TG_UTF8: {
            if (!offsets) throw Error(TG_ERR_INVALID_ARG, "Utf8 column requires offsets");
            const int32_t o0 = offsets[0], o1 = offsets[n];
            const int64_t nbytes = (int64_t)o1 - o0;
            if (nbytes < 0) throw Error(TG_ERR_INVALID_ARG, "Utf8 offsets are not monotonic");
            if (c.value_bytes + nbytes > INT32_MAX)
                throw Error(TG_ERR_UNSUPPORTED, "Utf8 column exceeds 2 GiB of value bytes (use LargeUtf8 sharding)");
            e.dev_reserve(c.values, (size_t)(c.value_bytes + nbytes), (size_t)c.value_bytes);
            e.h2d(c.values.p + c.value_bytes, (const uint8_t*)values + o0, (size_t)nbytes);
            // rebase offsets onto the concatenated byte buffer
            e.dev_reserve(c.offsets, (size_t)(have + n + 1) * 4, (size_t)(have + 1) * 4);
            std::vector<int32_t> tmp((size_t)n + 1);
            const int32_t delta = (int32_t)c.value_bytes - o0;
            for (int64_t i = 0; i <= n; ++i) tmp[i] = offsets[i] + delta;
            e.h2d(c.offsets.p + (size_t)have * 4, tmp.data(), (size_t)(n + 1) * 4);
            c.value_bytes += nbytes;
        } break;
        default: throw Error(TG_ERR_INVALID_ARG, "unknown dtype");
    }
    c.n_rows = have + n;
}

void table_append_host(Table& t, const std::string& name, int32_t dtype, int64_t n, const void* values,
                       const int32_t* offsets, const uint8_t* validity, int64_t bit_offset) {
    AppendTxn txn(t);
    append_host_column(txn, name, dtype, n, values, offsets, validity, bit_offset);
    txn.commit();
}

void table_adopt_device(Table& t, const std::string& name, int32_t dtype, int64_t n, const void* d_values,
                        const int32_t* d_offsets, const uint8_t* d_validity, int64_t n_value_bytes) {
    Engine& e = *t.eng;
    std::lock_guard<std::mutex> g(e.mu);
    TG_CUDA(cudaSetDevice(e.device));
    if (t.find(name)) throw Error(TG_ERR_INVALID_ARG, "column '" + name + "' already exists");
    if (((uintptr_t)d_values & 15) || ((uintptr_t)d_validity & 15) || ((uintptr_t)d_offsets & 15))
        throw Error(TG_ERR_INVALID_ARG, "adopted device buffers must be 16-byte aligned");
    Column& c = *table_get_or_add(t, name, dtype);
    c.adopted = true;
    c.n_rows = n;
    c.values.p = (uint8_t*)d_values;
    c.values.owned = false;
    c.values.cap = 0;
    c.validity.p = (uint8_t*)d_validity;
    c.validity.owned = false;
    c.offsets.p = (uint8_t*)d_offsets;
    c.offsets.owned = false;
    c.value_bytes = dtype == TG_UTF8 ? n_value_bytes : n * c.elem_bytes();
    c.null_count = -1;
    if ((dtype == TG_INT64 || dtype == TG_FLOAT64) && n > 0) {
        const int64_t head = std::min<int64_t>(n, 65536);
        std::vector<uint8_t> hv((size_t)head * 8), hb((size_t)(head + 7) / 8);
        TG_CUDA(cudaMemcpy(hv.data(), d_values, hv.size(), cudaMemcpyDeviceToHost));
        if (d_validity) TG_CUDA(cudaMemcpy(hb.data(), d_validity, hb.size(), cudaMemcpyDeviceToHost));
        set_pivot_host(c, dtype, head, hv.data(), d_validity ? hb.data() : nullptr, 0);
    }
    t.n_rows = std::max(t.n_rows, n);
}

// ---- Arrow C Data Interface (https://arrow.apache.org/docs/format/CDataInterface.html) ----
struct ArrowSchema {
    const char* format;
    const char* name;
    const char* metadata;
    int64_t flags;
    int64_t n_children;
    struct ArrowSchema** children;
    struct ArrowSchema* dictionary;
    void (*release)(struct ArrowSchema*);
    void* private_data;
};
struct ArrowArray {
    int64_t length;
    int64_t null_count;
    int64_t offset;
    int64_t n_buffers;
    int64_t n_children;
    const void** buffers;
    struct ArrowArray** children;
    struct ArrowArray* dictionary;
    void (*release)(struct ArrowArray*);
    void* private_data;
};

// Arrow C Data Interface format string -> the stored type; width / signedness of the delivered values when they are widened
// on the host; DataFusion's name of the delivered type (nullptr: it is the stored type)
struct ArrowFormat {
    int32_t dtype = 0;
    int src_w = 0;
    bool src_unsigned = false, temporal = false, large_offsets = false;
    const char* src_type = nullptr;
    char temporal_unit = 0;
};
static ArrowFormat arrow_format(const std::string& fmt, const char* column) {
    ArrowFormat f;
    auto starts = [&](const char* pre) { return fmt.compare(0, strlen(pre), pre) == 0; };
    if (fmt == "l") f.dtype = TG_INT64;
    else if (fmt == "g") f.dtype = TG_FLOAT64;
    else if (fmt == "u") f.dtype = TG_UTF8;
    else if (fmt == "U") f.dtype = TG_UTF8, f.large_offsets = true;
    else if (fmt == "i") f.dtype = TG_INT32;
    else if (fmt == "f") f.dtype = TG_FLOAT32;
    else if (fmt == "b") f.dtype = TG_BOOL;
    else if (fmt == "c") f.dtype = TG_INT32, f.src_w = 1, f.src_type = "Int8";
    else if (fmt == "C") f.dtype = TG_INT32, f.src_w = 1, f.src_unsigned = true, f.src_type = "UInt8";
    else if (fmt == "s") f.dtype = TG_INT32, f.src_w = 2, f.src_type = "Int16";
    else if (fmt == "S") f.dtype = TG_INT32, f.src_w = 2, f.src_unsigned = true, f.src_type = "UInt16";
    else if (fmt == "I") f.dtype = TG_INT64, f.src_w = 4, f.src_unsigned = true, f.src_type = "UInt32";
    else if (fmt == "L") f.dtype = TG_INT64, f.src_w = 8, f.src_unsigned = true, f.src_type = "UInt64";
    else if (fmt == "tdD") f.dtype = TG_INT32, f.temporal = true, f.src_type = "Date32", f.temporal_unit = 'D';
    else if (fmt == "tdm") f.dtype = TG_INT64, f.temporal = true, f.src_type = "Date64", f.temporal_unit = 'm';
    else if (fmt == "tts" || fmt == "ttm") f.dtype = TG_INT32, f.temporal = true, f.src_type = "Time32";
    else if (fmt == "ttu" || fmt == "ttn") f.dtype = TG_INT64, f.temporal = true, f.src_type = "Time64";
    else if (starts("tss:") || starts("tsm:") || starts("tsu:") || starts("tsn:"))
        f.dtype = TG_INT64, f.temporal = true, f.src_type = "Timestamp", f.temporal_unit = fmt[2];
    else if (fmt == "tDs" || fmt == "tDm" || fmt == "tDu" || fmt == "tDn") f.dtype = TG_INT64, f.temporal = true, f.src_type = "Duration";
    else throw Error(TG_ERR_UNSUPPORTED, std::string("Arrow format '") + fmt + "' of column '" + column + "' is not supported");
    return f;
}

// Declares the Arrow type a stored Int32 / Int64 column stands for when its values arrived already in the stored
// representation (Parquet chunks annotated DATE / TIME / TIMESTAMP / INT(8|16): the physical INT32 / INT64 values ARE the
// Arrow values): the typing rules of table_append_arrow then apply to it.
void declare_arrow_type(Column& c, const std::string& fmt) {
    const ArrowFormat f = arrow_format(fmt, c.name.c_str());
    if (f.dtype != c.dtype || f.large_offsets) throw Error(TG_ERR_TYPE_MISMATCH, "column '" + c.name + "' does not store Arrow format '" + fmt + "'");
    if (f.src_w == 4 || f.src_w == 8)  // UInt32 / UInt64 need a conversion of the stored values, not a label
        throw Error(TG_ERR_UNSUPPORTED, "column '" + c.name + "': Arrow format '" + fmt + "' cannot be declared on stored values");
    c.src_type = f.src_type;
    c.src_unsigned = f.src_unsigned;
    c.temporal = f.temporal;
    c.temporal_unit = f.temporal_unit;
}

void table_set_column_arrow_type(Table& t, const std::string& name, const std::string& fmt) {
    Engine& e = *t.eng;
    std::lock_guard<std::mutex> g(e.mu);
    Column* c = t.find(name);
    if (!c) throw Error(TG_ERR_COLUMN_NOT_FOUND, "Schema error: No field named " + name + ". Valid fields are " + t.valid_fields() + ".");
    declare_arrow_type(*c, fmt);
}

// ---- string dictionaries and Utf8View -> Utf8, decoded on the device ----
// A column delivered as dictionary<int*, utf8 | large_utf8> or as utf8_view is stored as the plain Utf8 column of its
// LOGICAL values (what DataFusion's string functions, comparisons, COUNT(DISTINCT) and GROUP BY see). What crosses PCIe is
// the encoded form: the dictionary's bytes and the rows' indices, or the views and their data buffers. A locate kernel
// turns every row into an entry {staging offset, length} (str_entries.cuh) and the Parquet BYTE_ARRAY tail writes the
// offsets and bytes. A row is NULL when its validity bit is clear or its index names a NULL dictionary value (Arrow's
// logical NULL); the index or view under a NULL row is never read. Malformed input (an index outside the dictionary, a
// view outside its data buffer) raises a flag and is clamped before any load: an error, never an out-of-bounds access.

__device__ __forceinline__ bool arrow_row_valid(const uint8_t* __restrict__ bits, uint64_t bit) {
    return !bits || ((__ldg(bits + (bit >> 3)) >> (bit & 7)) & 1);
}

// one warp per block: each valid row's index -> the dictionary value's entry; NULL rows get length 0
template <typename IndexT>
__global__ void __launch_bounds__(PQ_THREADS) arrow_dict_locate_kernel(const IndexT* __restrict__ idx, const uint8_t* __restrict__ bits, uint32_t bit_shift,
                                                                      const PqBlock* __restrict__ blocks, int64_t n_blocks,
                                                                      const uint64_t* __restrict__ dict_ents, uint64_t dict_count,
                                                                      uint64_t* __restrict__ row_ent, unsigned long long* __restrict__ block_bytes,
                                                                      uint32_t* __restrict__ err) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (PQ_THREADS / 32);
    for (int64_t b = (int64_t)blockIdx.x * (PQ_THREADS / 32) + (threadIdx.x >> 5); b < n_blocks; b += warps) {
        const PqBlock blk = blocks[b];
        unsigned long long total = 0;
        bool bad = false;
        for (uint32_t i = lane; i < blk.n_rows; i += 32) {
            const uint64_t r = (uint64_t)blk.first_row + i;
            uint64_t ent = 0;
            if (arrow_row_valid(bits, r + bit_shift)) {
                const int64_t v = (int64_t)__ldg(idx + r);  // (a UInt64 index of 2^63 or more reads as negative: out of range too)
                if (v < 0 || (uint64_t)v >= dict_count) bad = true;
                else ent = __ldg(dict_ents + v);
            }
            row_ent[r] = ent;
            total += ent >> 40;
        }
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) total += __shfl_xor_sync(0xffffffffu, total, m);
        if (lane == 0) block_bytes[b] = total;
        if (bad) atomicOr(err, STR_ERR_RANGE);
    }
}

// one warp per block: each valid row's 16-byte view -> the entry of its bytes: inline (length <= 12, the bytes sit in the
// staged view itself at +4) or in data buffer `buf` at `offset` (the buffer's staging offset from buf_base, bounds from
// buf_size); NULL rows get length 0
__global__ void __launch_bounds__(PQ_THREADS) arrow_view_locate_kernel(const uint4* __restrict__ views /* at staging offset 0 */, const uint8_t* __restrict__ bits,
                                                                      uint32_t bit_shift, const PqBlock* __restrict__ blocks, int64_t n_blocks,
                                                                      const uint64_t* __restrict__ buf_base, const uint64_t* __restrict__ buf_size,
                                                                      uint32_t n_bufs, uint64_t* __restrict__ row_ent,
                                                                      unsigned long long* __restrict__ block_bytes, uint32_t* __restrict__ err) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (PQ_THREADS / 32);
    for (int64_t b = (int64_t)blockIdx.x * (PQ_THREADS / 32) + (threadIdx.x >> 5); b < n_blocks; b += warps) {
        const PqBlock blk = blocks[b];
        unsigned long long total = 0;
        uint32_t flags = 0;
        for (uint32_t i = lane; i < blk.n_rows; i += 32) {
            const uint64_t r = (uint64_t)blk.first_row + i;
            uint64_t ent = 0;
            if (arrow_row_valid(bits, r + bit_shift)) {
                const uint4 v = __ldg(views + r);
                const int32_t len = (int32_t)v.x;
                if (len < 0) {
                    flags |= STR_ERR_RANGE;
                } else if ((uint32_t)len > PQ_STR_MAX_LEN) {
                    flags |= STR_ERR_LONG;
                } else if (len <= 12) {
                    ent = pq_str_ent(r * 16 + 4, (uint32_t)len);
                } else if (v.z >= n_bufs || (uint64_t)v.w + (uint32_t)len > __ldg(buf_size + v.z)) {
                    flags |= STR_ERR_RANGE;  // (buffer index and offset are unsigned here: a negative Int32 is out of range too)
                } else {
                    ent = pq_str_ent(__ldg(buf_base + v.z) + v.w, (uint32_t)len);
                }
            }
            row_ent[r] = ent;
            total += ent >> 40;
        }
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) total += __shfl_xor_sync(0xffffffffu, total, m);
        if (lane == 0) block_bytes[b] = total;
        if (flags) atomicOr(err, flags);
    }
}

namespace {

// One staging block per append: [payload | validity bits | blocks | tables | row entries | block totals | bases | flag].
// The caller fills payload and tables; the rest is laid out and uploaded here.
struct ArrowStage {
    uint8_t* p = nullptr;              // the block; the payload starts at p
    const uint8_t* bits = nullptr;     // staged validity (nullptr: no NULLs)
    uint8_t* tables = nullptr;         // the caller's lookup tables
    Utf8Entries x;
};

// validity: `bits` read from bit `bit_off` (nullptr: no NULLs); staged from its byte bit_off / 8 on
ArrowStage arrow_stage(Engine& e, size_t payload_b, size_t tables_b, int64_t n, const uint8_t* bits, int64_t bit_off, uint32_t* bit_shift) {
    ArrowStage s;
    const int64_t nb = (n + PQ_BLOCK_ROWS - 1) / PQ_BLOCK_ROWS;
    const size_t bits_n = bits ? (size_t)((bit_off & 7) + n + 7) / 8 : 0;
    const size_t pay_b = r16(payload_b), bits_b = r16(bits_n), blk_b = r16((size_t)nb * sizeof(PqBlock)), tab_b = r16(tables_b);
    const size_t re_b = r16((size_t)n * 8), bb_b = r16((size_t)(nb + 1) * 8);
    const size_t total = pay_b + bits_b + blk_b + tab_b + re_b + 2 * bb_b + 16 + 64;
    if (pay_b >= PQ_STAGE_MAX) throw Error(TG_ERR_UNSUPPORTED, "Arrow string batch of 1 TiB or more");
    s.p = e.dev_alloc(total);
    e.deferred_free.emplace_back(s.p, total);
    uint8_t* q = s.p + pay_b;
    if (bits) {
        e.h2d(q, bits + bit_off / 8, bits_n);
        s.bits = q;
    }
    *bit_shift = (uint32_t)(bits ? bit_off & 7 : 0);
    q += bits_b;
    std::vector<PqBlock> blocks((size_t)nb);
    for (int64_t b = 0; b < nb; ++b)
        blocks[(size_t)b] = PqBlock{0, (uint32_t)(b * PQ_BLOCK_ROWS), (uint32_t)std::min<int64_t>(PQ_BLOCK_ROWS, n - b * PQ_BLOCK_ROWS), 0u, 0u, 0u, 0u};
    e.h2d(q, blocks.data(), blocks.size() * sizeof(PqBlock));
    s.x.blocks = (const PqBlock*)q;
    s.x.n_blocks = nb;
    q += blk_b;
    s.tables = q;
    q += tab_b;
    s.x.row_ent = (const uint64_t*)q;
    q += re_b;
    s.x.block_bytes = (unsigned long long*)q;
    q += bb_b;
    s.x.block_base = (unsigned long long*)q;
    q += bb_b;
    s.x.err = (const uint32_t*)q;
    TG_CUDA(cudaMemsetAsync(q, 0, 4, e.copy_stream));
    s.x.stage = s.p;
    return s;
}

// the shared tail; a flag raised by the locate kernel becomes the error (and nothing was appended)
void arrow_utf8_finish(Engine& e, Column& c, const ArrowStage& s, int64_t n, const std::string& range_msg, const char* name) {
    const uint32_t err = append_utf8_from_entries(e, c, s.x, n);
    if (err & STR_ERR_RANGE) throw Error(TG_ERR_INVALID_ARG, std::string("column '") + name + "': " + range_msg);
    if (err & STR_ERR_LONG) throw Error(TG_ERR_UNSUPPORTED, std::string("column '") + name + "': string value of 16 MiB or more");
}

}  // namespace

// The entries of a string dictionary of dn values (host: it is small next to the rows), relative to the dictionary bytes'
// first byte d0, and per value "is valid" when one of them is NULL (empty otherwise). `offs` = its offsets from its own
// offset on (int64 when large_values), `dbits` its validity bitmap read from bit dbit0 (nullptr: no NULLs); host memory.
static void arrow_dict_entries(const char* name, bool large_values, int64_t dn, const void* offs, const uint8_t* dbits, int64_t dbit0,
                               std::vector<uint64_t>& ents, std::vector<uint8_t>& dict_valid, int64_t& d0, int64_t& d1) {
    ents.assign((size_t)dn, 0);
    dict_valid.clear();
    d0 = d1 = 0;
    if (dn == 0) return;
    auto o = [&](int64_t k) -> int64_t { return large_values ? ((const int64_t*)offs)[k] : (int64_t)((const int32_t*)offs)[k]; };
    d0 = o(0);
    d1 = o(dn);
    if (d1 < d0) throw Error(TG_ERR_INVALID_ARG, std::string("dictionary of column '") + name + "': offsets are not monotonic");
    dict_valid.assign((size_t)dn, 1);
    bool dict_nulls = false;
    for (int64_t k = 0; k < dn; ++k) {
        const int64_t a = o(k), b = o(k + 1);
        if (a < d0 || b < a || b > d1) throw Error(TG_ERR_INVALID_ARG, std::string("dictionary of column '") + name + "': offsets are not monotonic");
        if (b - a > (int64_t)PQ_STR_MAX_LEN) throw Error(TG_ERR_UNSUPPORTED, std::string("dictionary of column '") + name + "': string value of 16 MiB or more");
        const bool ok = !dbits || ((dbits[(dbit0 + k) >> 3] >> ((dbit0 + k) & 7)) & 1);
        dict_valid[(size_t)k] = ok;
        dict_nulls |= !ok;
        ents[(size_t)k] = ok ? pq_str_ent((uint64_t)(a - d0), (uint32_t)(b - a)) : 0;
    }
    if (!dict_nulls) dict_valid.clear();
}

static int arrow_index_width(char index_fmt) {
    return index_fmt == 'c' || index_fmt == 'C' ? 1 : index_fmt == 's' || index_fmt == 'S' ? 2 : index_fmt == 'i' || index_fmt == 'I' ? 4 : 8;
}

// dictionary<index fmt, utf8 | large_utf8>: `dict` is the dictionary child (its own offset and validity)
static void append_arrow_dict_utf8(AppendTxn& txn, const char* name, char index_fmt, bool large_values, const ArrowArray* ca, const ArrowArray* dict) {
    Engine& e = txn.e;
    Column& c = txn.column(name, TG_UTF8);
    const int64_t n = ca->length, off = ca->offset;
    if (n == 0) return;
    if (n >= ((int64_t)1 << 31)) throw Error(TG_ERR_UNSUPPORTED, std::string("column '") + name + "': a batch of 2^31 rows or more");
    const int iw = arrow_index_width(index_fmt);
    const bool idx_signed = index_fmt == 'c' || index_fmt == 's' || index_fmt == 'i' || index_fmt == 'l';
    const uint8_t* validity = ca->null_count == 0 ? nullptr : (const uint8_t*)ca->buffers[0];
    const uint8_t* idx = (const uint8_t*)ca->buffers[1] + off * iw;
    const int64_t dn = dict->length, doff = dict->offset;
    std::vector<uint64_t> ents;
    std::vector<uint8_t> dict_valid;
    int64_t d0 = 0, d1 = 0;
    arrow_dict_entries(name, large_values, dn, dn > 0 ? (const uint8_t*)dict->buffers[1] + doff * (large_values ? 8 : 4) : nullptr,
                       dict->null_count == 0 ? nullptr : (const uint8_t*)dict->buffers[0], doff, ents, dict_valid, d0, d1);
    // ---- a NULL dictionary value makes the rows naming it NULL: the rows' bitmap AND "index -> value valid", on the host
    std::vector<uint8_t> combined;
    int64_t bit_off = off;
    if (!dict_valid.empty()) {
        combined.assign((size_t)(n + 7) / 8, 0);
        for (int64_t r = 0; r < n; ++r) {
            if (validity && !((validity[(off + r) >> 3] >> ((off + r) & 7)) & 1)) continue;
            int64_t v;
            switch (iw) {
                case 1: v = idx_signed ? (int64_t)((const int8_t*)idx)[r] : (int64_t)idx[r]; break;
                case 2: v = idx_signed ? (int64_t)((const int16_t*)idx)[r] : (int64_t)((const uint16_t*)idx)[r]; break;
                case 4: v = idx_signed ? (int64_t)((const int32_t*)idx)[r] : (int64_t)((const uint32_t*)idx)[r]; break;
                default: v = ((const int64_t*)idx)[r]; break;
            }
            if (v < 0 || v >= dn) throw Error(TG_ERR_INVALID_ARG, std::string("dictionary column '") + name + "': an index lies outside the dictionary");
            if (dict_valid[(size_t)v]) combined[(size_t)(r >> 3)] |= (uint8_t)(1u << (r & 7));
        }
        validity = combined.data();
        bit_off = 0;
    }
    // ---- staging: dictionary bytes | indices | (validity, blocks, entries, ..)
    const size_t dict_b = r16((size_t)(d1 - d0)), idx_b = (size_t)n * iw;
    uint32_t bit_shift = 0;
    ArrowStage s = arrow_stage(e, dict_b + idx_b, (size_t)dn * 8, n, validity, bit_off, &bit_shift);
    if (d1 > d0) e.h2d(s.p, (const uint8_t*)dict->buffers[2] + d0, (size_t)(d1 - d0));
    e.h2d(s.p + dict_b, idx, idx_b);
    if (dn > 0) e.h2d(s.tables, ents.data(), (size_t)dn * 8);
    const uint64_t* d_ents = (const uint64_t*)s.tables;
    uint64_t* row = const_cast<uint64_t*>(s.x.row_ent);
    uint32_t* err = const_cast<uint32_t*>(s.x.err);
    const int grid = pq_str_grid(e, s.x.n_blocks);
    const uint8_t* d_idx = s.p + dict_b;
#define TG_DICT_LOCATE(T)                                                                                                           \
    arrow_dict_locate_kernel<T><<<grid, PQ_THREADS, 0, e.copy_stream>>>((const T*)d_idx, s.bits, bit_shift, s.x.blocks, s.x.n_blocks, d_ents, \
                                                                         (uint64_t)dn, row, s.x.block_bytes, err)
    switch (index_fmt) {
        case 'c': TG_DICT_LOCATE(int8_t); break;
        case 'C': TG_DICT_LOCATE(uint8_t); break;
        case 's': TG_DICT_LOCATE(int16_t); break;
        case 'S': TG_DICT_LOCATE(uint16_t); break;
        case 'i': TG_DICT_LOCATE(int32_t); break;
        case 'I': TG_DICT_LOCATE(uint32_t); break;
        case 'l': TG_DICT_LOCATE(int64_t); break;
        default: TG_DICT_LOCATE(uint64_t); break;
    }
#undef TG_DICT_LOCATE
    TG_CUDA(cudaGetLastError());
    e.launches += 1;
    const int64_t have = c.n_rows;
    arrow_utf8_finish(e, c, s, n, "a dictionary index lies outside the dictionary", name);
    append_validity(e, c, have, validity, bit_off, n);
}

// utf8_view: buffers = validity, views, data buffers.., variadic buffer sizes (int64 per data buffer)
static void append_arrow_view_utf8(AppendTxn& txn, const char* name, const ArrowArray* ca) {
    Engine& e = txn.e;
    Column& c = txn.column(name, TG_UTF8);
    const int64_t n = ca->length, off = ca->offset;
    if (n == 0) return;
    if (n >= ((int64_t)1 << 31)) throw Error(TG_ERR_UNSUPPORTED, std::string("column '") + name + "': a batch of 2^31 rows or more");
    if (ca->n_buffers < 3) throw Error(TG_ERR_INVALID_ARG, std::string("Utf8View column '") + name + "': expected a variadic buffer-sizes buffer");
    const int64_t n_data = ca->n_buffers - 3;
    if (n_data >= ((int64_t)1 << 32)) throw Error(TG_ERR_INVALID_ARG, std::string("Utf8View column '") + name + "': too many data buffers");
    const int64_t* sizes = (const int64_t*)ca->buffers[ca->n_buffers - 1];
    const uint8_t* validity = ca->null_count == 0 ? nullptr : (const uint8_t*)ca->buffers[0];
    // ---- staging: views | data buffers (16-byte aligned) | (validity, blocks, buffer bases + sizes, ..)
    const size_t views_b = r16((size_t)n * 16);
    std::vector<uint64_t> tab((size_t)n_data * 2);  // [base.. | size..]
    size_t pos = views_b;
    for (int64_t k = 0; k < n_data; ++k) {
        const int64_t sz = sizes ? sizes[k] : 0;
        if (sz < 0) throw Error(TG_ERR_INVALID_ARG, std::string("Utf8View column '") + name + "': negative data buffer size");
        tab[(size_t)k] = pos;
        tab[(size_t)(n_data + k)] = (uint64_t)sz;
        pos += r16((size_t)sz);
    }
    uint32_t bit_shift = 0;
    ArrowStage s = arrow_stage(e, pos, tab.size() * 8, n, validity, off, &bit_shift);
    e.h2d(s.p, (const uint8_t*)ca->buffers[1] + off * 16, (size_t)n * 16);
    for (int64_t k = 0; k < n_data; ++k)
        if (tab[(size_t)(n_data + k)]) e.h2d(s.p + tab[(size_t)k], ca->buffers[2 + k], (size_t)tab[(size_t)(n_data + k)]);
    if (!tab.empty()) e.h2d(s.tables, tab.data(), tab.size() * 8);
    const uint64_t* d_tab = (const uint64_t*)s.tables;
    arrow_view_locate_kernel<<<pq_str_grid(e, s.x.n_blocks), PQ_THREADS, 0, e.copy_stream>>>(
        (const uint4*)s.p, s.bits, bit_shift, s.x.blocks, s.x.n_blocks, d_tab, d_tab + n_data, (uint32_t)n_data,
        const_cast<uint64_t*>(s.x.row_ent), s.x.block_bytes, const_cast<uint32_t*>(s.x.err));
    TG_CUDA(cudaGetLastError());
    e.launches += 1;
    const int64_t have = c.n_rows;
    arrow_utf8_finish(e, c, s, n, "a Utf8View view lies outside its data buffer", name);
    append_validity(e, c, have, validity, off, n);
}

// the Arrow type of a dictionary's values as arrow-rs names it (for the refusal message)
static std::string arrow_type_name(const char* fmt) {
    static const char* const names[][2] = {{"z", "Binary"}, {"Z", "LargeBinary"}, {"vz", "BinaryView"}, {"vu", "Utf8View"}, {"b", "Boolean"},
                                           {"c", "Int8"}, {"C", "UInt8"}, {"s", "Int16"}, {"S", "UInt16"}, {"i", "Int32"}, {"I", "UInt32"},
                                           {"l", "Int64"}, {"L", "UInt64"}, {"e", "Float16"}, {"f", "Float32"}, {"g", "Float64"},
                                           {"u", "Utf8"}, {"U", "LargeUtf8"}, {"tdD", "Date32"}, {"tdm", "Date64"}};
    const std::string f = fmt ? fmt : "";
    for (const auto& n : names)
        if (f == n[0]) return n[1];
    return "Arrow format '" + f + "'";
}

void table_append_arrow(Table& t, const void* schema_p, const void* array_p) {
    const ArrowSchema* sc = (const ArrowSchema*)schema_p;
    const ArrowArray* ar = (const ArrowArray*)array_p;
    if (!sc || !ar || !sc->format || strcmp(sc->format, "+s") != 0)
        throw Error(TG_ERR_INVALID_ARG, "expected a struct-typed ArrowArray (a RecordBatch)");
    if (ar->offset != 0) throw Error(TG_ERR_UNSUPPORTED, "sliced struct arrays are not supported");
    AppendTxn txn(t);  // a child that fails undoes the children before it
    for (int64_t i = 0; i < sc->n_children; ++i) {
        const ArrowSchema* cs = sc->children[i];
        const ArrowArray* ca = ar->children[i];
        const std::string fmt = cs->format;
        if (cs->dictionary) {
            // dictionary<integer, utf8 | large_utf8>: decoded to the Utf8 column of the logical values; other value types are
            // refused (DataFusion's typing of MIN / MAX / SUM over numeric / temporal / Boolean dictionaries is not pinned)
            const char* vf = cs->dictionary->format;
            const bool int_index = fmt.size() == 1 && strchr("cCsSiIlL", fmt[0]) != nullptr;
            const bool utf8_values = vf && (strcmp(vf, "u") == 0 || strcmp(vf, "U") == 0);
            if (!int_index || !utf8_values || !ca->dictionary)
                throw Error(TG_ERR_UNSUPPORTED, std::string("column '") + cs->name + "': dictionary of " + arrow_type_name(vf) +
                                                    " values (index type " + arrow_type_name(fmt.c_str()) + ") is not supported; string dictionaries only");
            append_arrow_dict_utf8(txn, cs->name, fmt[0], vf[0] == 'U', ca, ca->dictionary);
            continue;
        }
        if (fmt == "vu") {
            append_arrow_view_utf8(txn, cs->name, ca);
            continue;
        }
        if (fmt == "vz") throw Error(TG_ERR_UNSUPPORTED, std::string("column '") + cs->name + "': BinaryView is not supported");
        const ArrowFormat F = arrow_format(fmt, cs->name);
        const int32_t dtype = F.dtype;
        const int src_w = F.src_w;
        const bool src_unsigned = F.src_unsigned, temporal = F.temporal, large_offsets = F.large_offsets;
        const char* src_type = F.src_type;
        const uint8_t* validity = (const uint8_t*)ca->buffers[0];
        if (ca->null_count == 0) validity = nullptr;
        const int64_t off = ca->offset, n = ca->length;
        if (src_type) {  // (checked before anything is appended: a column keeps one delivered type)
            Column* have = t.find(cs->name);
            if (have && (have->src_type == nullptr || strcmp(have->src_type, src_type) != 0))
                throw Error(TG_ERR_TYPE_MISMATCH, std::string("column '") + cs->name + "' was registered with a different type");
        }
        if (dtype == TG_UTF8 && large_offsets) {
            // LargeUtf8: 64-bit offsets narrowed on the host (a batch of 2 GiB or more of string bytes does not fit Utf8)
            const int64_t* o64 = (const int64_t*)ca->buffers[1] + off;
            std::vector<int32_t> o32((size_t)n + 1);
            const int64_t base = n > 0 || ca->buffers[1] ? o64[0] : 0;
            for (int64_t r = 0; r <= n; ++r) {
                const int64_t d = (ca->buffers[1] ? o64[r] : 0) - base;
                if (d > 0x7fffffffll) throw Error(TG_ERR_UNSUPPORTED, std::string("LargeUtf8 column '") + cs->name + "': a batch holds 2 GiB or more of string bytes");
                o32[(size_t)r] = (int32_t)d;
            }
            append_host_column(txn, cs->name, dtype, n, (const uint8_t*)ca->buffers[2] + base, o32.data(), validity, off);
        } else if (dtype == TG_UTF8) {
            const int32_t* offs = (const int32_t*)ca->buffers[1] + off;
            append_host_column(txn, cs->name, dtype, n, ca->buffers[2], offs, validity, off);
        } else if (dtype == TG_BOOL) {
            // values bitmap shares the array offset; append_bits takes one bit offset for both
            append_host_column(txn, cs->name, dtype, n, ca->buffers[1], nullptr, validity, off);
        } else if (src_w && src_w != (dtype == TG_INT64 ? 8 : 4)) {
            // Int8 / Int16 / UInt8 / UInt16 -> Int32, UInt32 -> Int64: widened exactly on the host
            const uint8_t* src = (const uint8_t*)ca->buffers[1] + off * src_w;
            std::vector<uint8_t> wide((size_t)n * (dtype == TG_INT64 ? 8 : 4));
            for (int64_t r = 0; r < n; ++r) {
                if (src_w == 1) {
                    const int32_t v = src_unsigned ? (int32_t)src[r] : (int32_t)(int8_t)src[r];
                    memcpy(wide.data() + r * 4, &v, 4);
                } else if (src_w == 2) {
                    uint16_t u;
                    memcpy(&u, src + r * 2, 2);
                    const int32_t v = src_unsigned ? (int32_t)u : (int32_t)(int16_t)u;
                    memcpy(wide.data() + r * 4, &v, 4);
                } else {
                    uint32_t u;
                    memcpy(&u, src + r * 4, 4);
                    const int64_t v = (int64_t)u;
                    memcpy(wide.data() + r * 8, &v, 8);
                }
            }
            append_host_column(txn, cs->name, dtype, n, wide.data(), nullptr, validity, off);
        } else {
            const int w = dtype == TG_INT64 || dtype == TG_FLOAT64 ? 8 : 4;
            const uint8_t* vals = (const uint8_t*)ca->buffers[1] + off * w;
            if (src_unsigned && src_w == 8) {  // UInt64: representable as Int64 unless a valid value has the top bit set
                for (int64_t r = 0; r < n; ++r) {
                    if (validity && !((validity[(off + r) >> 3] >> ((off + r) & 7)) & 1)) continue;
                    if (vals[r * 8 + 7] & 0x80) throw Error(TG_ERR_UNSUPPORTED, std::string("UInt64 column '") + cs->name + "' holds values above the Int64 range");
                }
            }
            append_host_column(txn, cs->name, dtype, n, vals, nullptr, validity, off);
        }
        if (src_type) {
            Column* c = t.find(cs->name);
            c->src_type = src_type;
            c->src_unsigned = src_unsigned;
            c->temporal = temporal;
            c->temporal_unit = F.temporal_unit;
        }
    }
    txn.commit();
}

// ---- Arrow C Device Data Interface (https://arrow.apache.org/docs/format/CDeviceDataInterface.html) ----
// A RecordBatch whose buffers are in HBM is appended by copies and kernels on the device: it leaves exactly the state that
// table_append_arrow leaves for the same batch in host memory (buffers, NULL counts, pivots, tail mirrors, delivered types,
// errors). Nothing crosses PCIe but the small read-backs named below.
struct ArrowDeviceArray {
    ArrowArray array;
    int64_t device_id;
    int32_t device_type;
    void* sync_event;
    int64_t reserved[3];
};
static_assert(sizeof(ArrowDeviceArray) == 128 && offsetof(ArrowDeviceArray, device_type) == 88 && offsetof(ArrowDeviceArray, sync_event) == 96,
              "ArrowDeviceArray layout");
constexpr int32_t ARROW_DEVICE_CPU = 1, ARROW_DEVICE_CUDA = 2, ARROW_DEVICE_CUDA_HOST = 3, ARROW_DEVICE_CUDA_MANAGED = 13;

// what the kernels of one column report; read back once per batch
struct ArrowDevResult {
    unsigned long long zeros;    // clear bits of the column's validity (its NULL rows)
    unsigned long long last64;   // validity bits of rows n - 64 .. n - 1 (bit k: row n - 64 + k)
    unsigned long long vlast64;  // the same for Boolean values
    uint32_t flags;              // ARROW_DEV_ERR_*
    uint32_t pad;
};
constexpr uint32_t ARROW_DEV_ERR_U64 = 1u;    // a valid UInt64 value of 2^63 or more
constexpr uint32_t ARROW_DEV_ERR_LARGE = 2u;  // a LargeUtf8 offset 2 GiB or more past the batch's first
constexpr uint32_t ARROW_DEV_ERR_DICT = 4u;   // (in the locate kernel's flag word) a valid row's index outside the dictionary

__device__ __forceinline__ uint64_t grid_thread() { return (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; }
__device__ __forceinline__ uint64_t grid_threads() { return (uint64_t)gridDim.x * blockDim.x; }

// bits [s, s + len) (1 <= len <= 32) of the LSB-first bitmap `src` (4-byte aligned); loads only words that hold one of them
__device__ __forceinline__ uint32_t arrow_bits32(const uint32_t* __restrict__ src, uint64_t s, uint32_t len) {
    const uint32_t sh = (uint32_t)(s & 31);
    const uint32_t lo = __ldg(src + (s >> 5));
    const uint32_t hi = sh + len > 32 ? __ldg(src + (s >> 5) + 1) : 0u;
    const uint32_t v = __funnelshift_r(lo, hi, sh);
    return len < 32 ? v & ((1u << len) - 1u) : v;
}

// stores word w of an n-row chunk-relative bitmap (bits past n clear) and ORs its share of the last 64 rows into *last64
__device__ __forceinline__ void arrow_word_out(uint32_t* __restrict__ out, uint64_t w, uint32_t v, uint64_t n, unsigned long long* last64) {
    out[w] = v;
    const int64_t sh = 32 * (int64_t)w - ((int64_t)n - 64);
    if (v && sh > -32) atomicOr(last64, sh >= 0 ? (unsigned long long)v << sh : (unsigned long long)v >> -sh);
}

__device__ __forceinline__ void arrow_add_zeros(unsigned long long* zeros, unsigned long long z) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) z += __shfl_xor_sync(0xffffffffu, z, m);
    if ((threadIdx.x & 31) == 0 && z) atomicAdd(zeros, z);
}

// bits [bit0, bit0 + n) of a producer's bitmap -> chunk-relative 32-bit words, their clear bits (zeros may be nullptr) and
// the last 64 bits; the input of append_validity_device / append_bits_device
__global__ void __launch_bounds__(256) arrow_bits_extract_kernel(const uint32_t* __restrict__ src, uint64_t bit0, uint64_t n, uint32_t* __restrict__ out,
                                                                 unsigned long long* zeros, unsigned long long* last64) {
    const uint64_t n_words = (n + 31) / 32;
    unsigned long long z = 0;
    // (every warp runs the same number of rounds: the shuffle in arrow_add_zeros needs all 32 lanes)
    const uint64_t rounds = (n_words + grid_threads() - 1) / grid_threads();
    for (uint64_t k = 0; k < rounds; ++k) {
        const uint64_t w = grid_thread() + k * grid_threads();
        if (w >= n_words) continue;
        const uint32_t len = (uint32_t)(n - 32 * w < 32 ? n - 32 * w : 32);
        const uint32_t v = arrow_bits32(src, bit0 + 32 * w, len);
        arrow_word_out(out, w, v, n, last64);
        z += len - __popc(v);
    }
    if (zeros) arrow_add_zeros(zeros, z);
}

// Int8 / UInt8 / Int16 / UInt16 -> Int32, UInt32 -> Int64, exactly
template <typename S, typename D>
__global__ void __launch_bounds__(256) arrow_widen_kernel(const S* __restrict__ src, D* __restrict__ dst, uint64_t n) {
    for (uint64_t i = grid_thread(); i < n; i += grid_threads()) dst[i] = (D)__ldg(src + i);
}

// UInt64 -> Int64: copied as they are; a VALID value with the top bit set raises ARROW_DEV_ERR_U64
__global__ void __launch_bounds__(256) arrow_u64_kernel(const uint64_t* __restrict__ src, uint64_t* __restrict__ dst, uint64_t n,
                                                        const uint8_t* __restrict__ bits, uint64_t bit0, uint32_t* flags) {
    bool bad = false;
    for (uint64_t i = grid_thread(); i < n; i += grid_threads()) {
        const uint64_t v = __ldg(src + i);
        dst[i] = v;
        if ((v >> 63) && arrow_row_valid(bits, bit0 + i)) bad = true;
    }
    if (bad) atomicOr(flags, ARROW_DEV_ERR_U64);
}

// n + 1 Utf8 / LargeUtf8 offsets rebased onto the column's bytes: out[i] = (int32)(src[i] - first) + byte_base, in 32-bit
// arithmetic as the host path does; LargeUtf8 (check) flags an offset 2 GiB or more past the first
template <typename O>
__global__ void __launch_bounds__(256) arrow_offsets_kernel(const O* __restrict__ src, int32_t* __restrict__ dst, uint64_t n1, int64_t first,
                                                            uint32_t byte_base, bool check, uint32_t* flags) {
    bool bad = false;
    for (uint64_t i = grid_thread(); i < n1; i += grid_threads()) {
        const int64_t d = (int64_t)__ldg(src + i) - first;
        bad |= check && d > 0x7fffffffll;
        dst[i] = (int32_t)((uint32_t)d + byte_base);
    }
    if (bad) atomicOr(flags, ARROW_DEV_ERR_LARGE);
}

// a dictionary holding a NULL value: row valid AND its value valid, as chunk-relative words (+ clear bits, last 64 bits); a
// valid row's index outside the dictionary raises ARROW_DEV_ERR_DICT and is never used to load
template <typename IndexT>
__global__ void __launch_bounds__(256) arrow_dict_valid_kernel(const IndexT* __restrict__ idx, const uint8_t* __restrict__ bits, uint64_t bit0, uint64_t n,
                                                               const uint8_t* __restrict__ dict_valid, uint64_t dn, uint32_t* __restrict__ out,
                                                               unsigned long long* zeros, unsigned long long* last64, uint32_t* flags) {
    const uint64_t n_words = (n + 31) / 32;
    unsigned long long z = 0;
    bool bad = false;
    const uint64_t rounds = (n_words + grid_threads() - 1) / grid_threads();
    for (uint64_t k = 0; k < rounds; ++k) {
        const uint64_t w = grid_thread() + k * grid_threads();
        if (w >= n_words) continue;
        const uint32_t len = (uint32_t)(n - 32 * w < 32 ? n - 32 * w : 32);
        uint32_t v = 0;
        for (uint32_t j = 0; j < len; ++j) {
            const uint64_t r = 32 * w + j;
            if (!arrow_row_valid(bits, bit0 + r)) continue;
            const int64_t x = (int64_t)__ldg(idx + r);  // (a UInt64 index of 2^63 or more reads as negative: out of range too)
            if (x < 0 || (uint64_t)x >= dn) bad = true;
            else v |= (uint32_t)__ldg(dict_valid + x) << j;
        }
        arrow_word_out(out, w, v, n, last64);
        z += len - __popc(v);
    }
    arrow_add_zeros(zeros, z);
    if (bad) atomicOr(flags, ARROW_DEV_ERR_DICT);
}

namespace {

int dev_grid(const Engine& e, uint64_t items) {
    return (int)std::max<uint64_t>(1, std::min<uint64_t>((items + 255) / 256, (uint64_t)e.sm_count * 8));
}

// a producer's bitmap read from bit `bit0`, as a 4-byte aligned base and the bit offset from it
struct DevBits {
    const uint32_t* base;
    uint64_t bit0;
};
DevBits dev_bits(const void* p, int64_t bit0) {
    const uintptr_t a = (uintptr_t)p;
    return DevBits{(const uint32_t*)(a & ~(uintptr_t)3), (uint64_t)bit0 + 8 * (a & 3)};
}

// one child of the batch between the kernels that read the producer's buffers and the merges that follow the read-back
struct DevChild {
    Column* c = nullptr;
    std::string name;
    int64_t have = 0, n = 0;
    uint32_t* vwords = nullptr;  // extracted validity (nullptr: the child delivers no bitmap)
    uint32_t* bwords = nullptr;  // extracted Boolean values
    const uint8_t* pivot_bits = nullptr;  // producer validity of the rows the pivot is taken from, read from bit pivot_bit0
    int64_t pivot_bit0 = 0;
    bool pivot = false;
};

struct DevBatch {
    Engine& e;
    ArrowDevResult* d_res = nullptr;  // [children]
    std::vector<DevChild> ch;

    uint32_t* words(int64_t n) {  // a chunk-relative bitmap of n rows, freed with the batch's other staging
        const size_t b = r16((size_t)(n + 31) / 32 * 4);
        uint8_t* p = e.dev_alloc(b);
        e.deferred_free.emplace_back(p, b);
        return (uint32_t*)p;
    }
    // validity of child i from the producer's bitmap (nullptr: no NULLs) -> words, zeros and last 64 bits in d_res[i]
    void extract_validity(size_t i, const void* bits, int64_t bit0) {
        DevChild& k = ch[i];
        if (!bits || k.n == 0) return;
        k.vwords = words(k.n);
        const DevBits b = dev_bits(bits, bit0);
        arrow_bits_extract_kernel<<<dev_grid(e, (uint64_t)(k.n + 31) / 32), 256, 0, e.copy_stream>>>(b.base, b.bit0, (uint64_t)k.n, k.vwords,
                                                                                                     &d_res[i].zeros, &d_res[i].last64);
        TG_CUDA(cudaGetLastError());
        e.launches += 1;
    }
    // the read-back of every child's result record so far (one copy, one synchronisation); the first raised flag is the error
    std::vector<ArrowDevResult> read_back(size_t upto) {
        std::vector<ArrowDevResult> r(upto);
        if (upto == 0) return r;
        ArrowDevResult* h = (ArrowDevResult*)e.host_scratch(upto * sizeof(ArrowDevResult));
        TG_CUDA(cudaMemcpyAsync(h, d_res, upto * sizeof(ArrowDevResult), cudaMemcpyDeviceToHost, e.copy_stream));
        TG_CUDA(cudaStreamSynchronize(e.copy_stream));
        memcpy(r.data(), h, upto * sizeof(ArrowDevResult));
        for (size_t i = 0; i < upto; ++i) {
            if (r[i].flags & ARROW_DEV_ERR_U64)
                throw Error(TG_ERR_UNSUPPORTED, "UInt64 column '" + ch[i].name + "' holds values above the Int64 range");
            if (r[i].flags & ARROW_DEV_ERR_LARGE)
                throw Error(TG_ERR_UNSUPPORTED, "LargeUtf8 column '" + ch[i].name + "': a batch holds 2 GiB or more of string bytes");
        }
        return r;
    }
};

// small device -> host read-backs (string offsets' end points, a dictionary's offsets and validity, Utf8View sizes)
void dev_read(Engine& e, void* dst, const void* src, size_t bytes) {
    if (bytes) TG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, e.copy_stream));
}

// buffer k of `a`, which a copy or kernel reads when the array has rows: a missing one is an error, not a load from address 0
void dev_need(const ArrowArray* a, int64_t k, const char* col) {
    if (a->length > 0 && (a->n_buffers <= k || !a->buffers[k]))
        throw Error(TG_ERR_INVALID_ARG, std::string("column '") + col + "': buffer " + std::to_string(k) + " of a CUDA device array is missing");
}

void dev_check_aligned(const void* p, size_t a, const std::string& what) {
    if ((uintptr_t)p % a) throw Error(TG_ERR_INVALID_ARG, what + " is not aligned to its " + std::to_string(a) + "-byte elements");
}

// every buffer of a child the device path reads must be device or managed memory of the engine's device
void dev_check_buffer(const Engine& e, const void* p, const char* col) {
    if (!p) return;
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        a.type = cudaMemoryTypeUnregistered;
    }
    if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged)
        throw Error(TG_ERR_INVALID_ARG, std::string("column '") + col + "': a buffer of a CUDA device array is not device memory");
    if (a.device != e.device)
        throw Error(TG_ERR_INVALID_ARG, std::string("column '") + col + "': a buffer of a CUDA device array lies on device " + std::to_string(a.device) +
                                            ", not on the engine's device " + std::to_string(e.device));
}

void dev_check_child(const Engine& e, const ArrowSchema* cs, const ArrowArray* ca) {
    const bool view = cs->format && strcmp(cs->format, "vu") == 0 && !cs->dictionary;
    for (int64_t b = 0; b < ca->n_buffers; ++b)
        if (!(view && b == ca->n_buffers - 1)) dev_check_buffer(e, ca->buffers[b], cs->name);  // (Utf8View sizes: read wherever they are)
    if (ca->dictionary)
        for (int64_t b = 0; b < ca->dictionary->n_buffers; ++b) dev_check_buffer(e, ca->dictionary->buffers[b], cs->name);
}

}  // namespace

// dictionary<index fmt, utf8 | large_utf8> on the device: the dictionary's offsets and validity are read back (small) for the
// host's entry table; the locate kernel reads the producer's indices, validity and dictionary bytes where they are
static void append_dev_dict_utf8(AppendTxn& txn, DevBatch& B, size_t i, char index_fmt, bool large_values, const ArrowArray* ca, const ArrowArray* dict) {
    Engine& e = txn.e;
    DevChild& k = B.ch[i];
    const char* name = k.name.c_str();
    Column& c = txn.column(k.name, TG_UTF8);
    k.c = &c;
    k.have = c.n_rows;
    const int64_t n = ca->length, off = ca->offset;
    if (n == 0) return;
    if (n >= ((int64_t)1 << 31)) throw Error(TG_ERR_UNSUPPORTED, std::string("column '") + name + "': a batch of 2^31 rows or more");
    const int iw = arrow_index_width(index_fmt);
    dev_need(ca, 1, name);
    dev_need(dict, 1, name);
    const uint8_t* validity = ca->null_count == 0 ? nullptr : (const uint8_t*)ca->buffers[0];
    const uint8_t* idx = (const uint8_t*)ca->buffers[1] + off * iw;
    dev_check_aligned(idx, (size_t)iw, std::string("the index buffer of column '") + name + "'");
    const int64_t dn = dict->length, doff = dict->offset;
    const int ow = large_values ? 8 : 4;
    std::vector<uint8_t> h_offs(dn > 0 ? (size_t)(dn + 1) * ow : 0), h_bits;
    const uint8_t* dbits = dict->null_count == 0 ? nullptr : (const uint8_t*)dict->buffers[0];
    if (dn > 0) {
        dev_read(e, h_offs.data(), (const uint8_t*)dict->buffers[1] + doff * ow, h_offs.size());
        if (dbits) {
            h_bits.resize((size_t)((doff & 7) + dn + 7) / 8);
            dev_read(e, h_bits.data(), dbits + doff / 8, h_bits.size());
        }
        TG_CUDA(cudaStreamSynchronize(e.copy_stream));
    }
    std::vector<uint64_t> ents;
    std::vector<uint8_t> dict_valid;
    int64_t d0 = 0, d1 = 0;
    arrow_dict_entries(name, large_values, dn, h_offs.data(), dbits ? h_bits.data() : nullptr, doff & 7, ents, dict_valid, d0, d1);
    if (d1 > d0 && (dict->n_buffers < 3 || !dict->buffers[2]))
        throw Error(TG_ERR_INVALID_ARG, std::string("column '") + name + "': the dictionary's data buffer is missing");
    uint32_t bit_shift = 0;
    ArrowStage s = arrow_stage(e, 0, (size_t)dn * 8 + (size_t)dn, n, nullptr, 0, &bit_shift);
    s.x.stage = (const uint8_t*)dict->buffers[2] + d0;
    if (dn > 0) e.h2d(s.tables, ents.data(), (size_t)dn * 8);
    uint32_t* err = const_cast<uint32_t*>(s.x.err);
    if (validity) {
        s.bits = validity + off / 8;
        bit_shift = (uint32_t)(off & 7);
    }
    if (!dict_valid.empty()) {
        // a NULL dictionary value makes the rows naming it NULL: the locate kernel and the column read the combined bitmap
        uint8_t* d_valid = s.tables + (size_t)dn * 8;
        e.h2d(d_valid, dict_valid.data(), (size_t)dn);
        k.vwords = B.words(n);
        const int g = dev_grid(e, (uint64_t)(n + 31) / 32);
#define TG_DICT_VALID(T)                                                                                                           \
    arrow_dict_valid_kernel<T><<<g, 256, 0, e.copy_stream>>>((const T*)idx, validity, (uint64_t)off, (uint64_t)n, d_valid, (uint64_t)dn, k.vwords, \
                                                             &B.d_res[i].zeros, &B.d_res[i].last64, err)
        switch (index_fmt) {
            case 'c': TG_DICT_VALID(int8_t); break;
            case 'C': TG_DICT_VALID(uint8_t); break;
            case 's': TG_DICT_VALID(int16_t); break;
            case 'S': TG_DICT_VALID(uint16_t); break;
            case 'i': TG_DICT_VALID(int32_t); break;
            case 'I': TG_DICT_VALID(uint32_t); break;
            case 'l': TG_DICT_VALID(int64_t); break;
            default: TG_DICT_VALID(uint64_t); break;
        }
#undef TG_DICT_VALID
        TG_CUDA(cudaGetLastError());
        e.launches += 1;
        s.bits = (const uint8_t*)k.vwords;
        bit_shift = 0;
    } else {
        B.extract_validity(i, validity, off);
    }
    const int grid = pq_str_grid(e, s.x.n_blocks);
#define TG_DICT_LOCATE(T)                                                                                                           \
    arrow_dict_locate_kernel<T><<<grid, PQ_THREADS, 0, e.copy_stream>>>((const T*)idx, s.bits, bit_shift, s.x.blocks, s.x.n_blocks, \
                                                                         (const uint64_t*)s.tables, (uint64_t)dn, const_cast<uint64_t*>(s.x.row_ent), \
                                                                         s.x.block_bytes, err)
    switch (index_fmt) {
        case 'c': TG_DICT_LOCATE(int8_t); break;
        case 'C': TG_DICT_LOCATE(uint8_t); break;
        case 's': TG_DICT_LOCATE(int16_t); break;
        case 'S': TG_DICT_LOCATE(uint16_t); break;
        case 'i': TG_DICT_LOCATE(int32_t); break;
        case 'I': TG_DICT_LOCATE(uint32_t); break;
        case 'l': TG_DICT_LOCATE(int64_t); break;
        default: TG_DICT_LOCATE(uint64_t); break;
    }
#undef TG_DICT_LOCATE
    TG_CUDA(cudaGetLastError());
    e.launches += 1;
    const uint32_t f = append_utf8_from_entries(e, c, s.x, n);
    if (f & ARROW_DEV_ERR_DICT) throw Error(TG_ERR_INVALID_ARG, std::string("dictionary column '") + name + "': an index lies outside the dictionary");
    if (f & STR_ERR_RANGE) throw Error(TG_ERR_INVALID_ARG, std::string("column '") + name + "': a dictionary index lies outside the dictionary");
    if (f & STR_ERR_LONG) throw Error(TG_ERR_UNSUPPORTED, std::string("column '") + name + "': string value of 16 MiB or more");
}

// utf8_view on the device: views and data buffers staged device to device, the locate kernel unchanged
static void append_dev_view_utf8(AppendTxn& txn, DevBatch& B, size_t i, const ArrowArray* ca) {
    Engine& e = txn.e;
    DevChild& k = B.ch[i];
    const char* name = k.name.c_str();
    Column& c = txn.column(k.name, TG_UTF8);
    k.c = &c;
    k.have = c.n_rows;
    const int64_t n = ca->length, off = ca->offset;
    if (n == 0) return;
    if (n >= ((int64_t)1 << 31)) throw Error(TG_ERR_UNSUPPORTED, std::string("column '") + name + "': a batch of 2^31 rows or more");
    if (ca->n_buffers < 3) throw Error(TG_ERR_INVALID_ARG, std::string("Utf8View column '") + name + "': expected a variadic buffer-sizes buffer");
    const int64_t n_data = ca->n_buffers - 3;
    if (n_data >= ((int64_t)1 << 32)) throw Error(TG_ERR_INVALID_ARG, std::string("Utf8View column '") + name + "': too many data buffers");
    dev_need(ca, 1, name);
    const void* d_sizes = ca->buffers[ca->n_buffers - 1];
    std::vector<int64_t> sizes((size_t)n_data, 0);
    if (d_sizes && n_data > 0) {
        cudaPointerAttributes a{};
        if (cudaPointerGetAttributes(&a, d_sizes) != cudaSuccess) {
            cudaGetLastError();
            a.type = cudaMemoryTypeUnregistered;
        }
        if (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) {
            dev_check_buffer(e, d_sizes, name);
            dev_read(e, sizes.data(), d_sizes, (size_t)n_data * 8);
            TG_CUDA(cudaStreamSynchronize(e.copy_stream));
        } else {
            memcpy(sizes.data(), d_sizes, (size_t)n_data * 8);
        }
    }
    const uint8_t* validity = ca->null_count == 0 ? nullptr : (const uint8_t*)ca->buffers[0];
    const size_t views_b = r16((size_t)n * 16);
    std::vector<uint64_t> tab((size_t)n_data * 2);  // [base.. | size..]
    size_t pos = views_b;
    for (int64_t j = 0; j < n_data; ++j) {
        const int64_t sz = sizes[(size_t)j];
        if (sz < 0) throw Error(TG_ERR_INVALID_ARG, std::string("Utf8View column '") + name + "': negative data buffer size");
        if (sz > 0 && !ca->buffers[2 + j]) throw Error(TG_ERR_INVALID_ARG, std::string("Utf8View column '") + name + "': a data buffer is missing");
        tab[(size_t)j] = pos;
        tab[(size_t)(n_data + j)] = (uint64_t)sz;
        pos += r16((size_t)sz);
    }
    uint32_t bit_shift = 0;
    ArrowStage s = arrow_stage(e, pos, tab.size() * 8, n, nullptr, 0, &bit_shift);
    TG_CUDA(cudaMemcpyAsync(s.p, (const uint8_t*)ca->buffers[1] + off * 16, (size_t)n * 16, cudaMemcpyDefault, e.copy_stream));
    for (int64_t j = 0; j < n_data; ++j)
        if (tab[(size_t)(n_data + j)])
            TG_CUDA(cudaMemcpyAsync(s.p + tab[(size_t)j], ca->buffers[2 + j], (size_t)tab[(size_t)(n_data + j)], cudaMemcpyDefault, e.copy_stream));
    if (!tab.empty()) e.h2d(s.tables, tab.data(), tab.size() * 8);
    if (validity) {
        s.bits = validity + off / 8;
        bit_shift = (uint32_t)(off & 7);
    }
    B.extract_validity(i, validity, off);
    const uint64_t* d_tab = (const uint64_t*)s.tables;
    arrow_view_locate_kernel<<<pq_str_grid(e, s.x.n_blocks), PQ_THREADS, 0, e.copy_stream>>>(
        (const uint4*)s.p, s.bits, bit_shift, s.x.blocks, s.x.n_blocks, d_tab, d_tab + n_data, (uint32_t)n_data,
        const_cast<uint64_t*>(s.x.row_ent), s.x.block_bytes, const_cast<uint32_t*>(s.x.err));
    TG_CUDA(cudaGetLastError());
    e.launches += 1;
    arrow_utf8_finish(e, c, s, n, "a Utf8View view lies outside its data buffer", name);
}

// one plain child (the formats of arrow_format) on the device; its validity / Boolean merges wait for the batch's read-back
static void append_dev_plain(AppendTxn& txn, DevBatch& B, size_t i, const ArrowFormat& F, const ArrowArray* ca) {
    Engine& e = txn.e;
    DevChild& k = B.ch[i];
    const std::string& name = k.name;
    const int32_t dtype = F.dtype;
    const uint8_t* validity = ca->null_count == 0 ? nullptr : (const uint8_t*)ca->buffers[0];
    const int64_t off = ca->offset, n = ca->length;
    if (n < 0) throw Error(TG_ERR_INVALID_ARG, "negative row count");
    Column& c = txn.column(name, dtype);
    k.c = &c;
    k.have = c.n_rows;
    if (n == 0) return;
    dev_need(ca, 1, name.c_str());
    const int64_t have = c.n_rows;
    const int g = dev_grid(e, (uint64_t)n);
    uint32_t* flags = &B.d_res[i].flags;
    if (dtype == TG_UTF8) {
        // the offsets' end points decide the byte count and are checked before anything is copied
        const int ow = F.large_offsets ? 8 : 4;
        const uint8_t* ob = (const uint8_t*)ca->buffers[1] + off * ow;
        dev_check_aligned(ob, (size_t)ow, "the offsets of column '" + name + "'");
        int64_t ends[2] = {0, 0};
        dev_read(e, &ends[0], ob, (size_t)ow);
        dev_read(e, &ends[1], ob + n * ow, (size_t)ow);
        TG_CUDA(cudaStreamSynchronize(e.copy_stream));
        if (ow == 4) ends[0] = (int32_t)ends[0], ends[1] = (int32_t)ends[1];
        int64_t nbytes = ends[1] - ends[0];
        if (F.large_offsets) {
            if (nbytes > 0x7fffffffll) throw Error(TG_ERR_UNSUPPORTED, "LargeUtf8 column '" + name + "': a batch holds 2 GiB or more of string bytes");
            nbytes = (int32_t)nbytes;  // (the host path narrows every offset to 32 bits first)
        }
        B.extract_validity(i, validity, off);
        if (nbytes < 0) throw Error(TG_ERR_INVALID_ARG, "Utf8 offsets are not monotonic");
        if (c.value_bytes + nbytes > INT32_MAX) throw Error(TG_ERR_UNSUPPORTED, "Utf8 column exceeds 2 GiB of value bytes (use LargeUtf8 sharding)");
        if (nbytes > 0) dev_need(ca, 2, name.c_str());
        e.dev_reserve(c.values, (size_t)(c.value_bytes + nbytes), (size_t)c.value_bytes);
        if (nbytes)
            TG_CUDA(cudaMemcpyAsync(c.values.p + c.value_bytes, (const uint8_t*)ca->buffers[2] + ends[0], (size_t)nbytes, cudaMemcpyDefault, e.copy_stream));
        e.dev_reserve(c.offsets, (size_t)(have + n + 1) * 4, (size_t)(have + 1) * 4);
        int32_t* dst = (int32_t*)c.offsets.p + have;
        const int go = dev_grid(e, (uint64_t)n + 1);
        if (F.large_offsets)
            arrow_offsets_kernel<int64_t><<<go, 256, 0, e.copy_stream>>>((const int64_t*)ob, dst, (uint64_t)n + 1, ends[0], (uint32_t)c.value_bytes, true, flags);
        else
            arrow_offsets_kernel<int32_t><<<go, 256, 0, e.copy_stream>>>((const int32_t*)ob, dst, (uint64_t)n + 1, ends[0], (uint32_t)c.value_bytes, false, flags);
        TG_CUDA(cudaGetLastError());
        e.launches += 1;
        c.value_bytes += nbytes;
    } else if (dtype == TG_BOOL) {
        B.extract_validity(i, validity, off);
        k.bwords = B.words(n);
        const DevBits b = dev_bits(ca->buffers[1], off);
        arrow_bits_extract_kernel<<<dev_grid(e, (uint64_t)(n + 31) / 32), 256, 0, e.copy_stream>>>(b.base, b.bit0, (uint64_t)n, k.bwords, nullptr,
                                                                                                   &B.d_res[i].vlast64);
        TG_CUDA(cudaGetLastError());
        e.launches += 1;
    } else {
        const size_t w = (size_t)c.elem_bytes();
        e.dev_reserve(c.values, (size_t)(have + n) * w, (size_t)have * w);
        uint8_t* dst = c.values.p + (size_t)have * w;
        const uint8_t* src = (const uint8_t*)ca->buffers[1];
        if (F.src_w && F.src_w != (int)w) {
            dev_check_aligned(src, (size_t)F.src_w, "the values of column '" + name + "'");
            if (F.src_w == 1 && F.src_unsigned) arrow_widen_kernel<uint8_t, int32_t><<<g, 256, 0, e.copy_stream>>>(src + off, (int32_t*)dst, (uint64_t)n);
            else if (F.src_w == 1) arrow_widen_kernel<int8_t, int32_t><<<g, 256, 0, e.copy_stream>>>((const int8_t*)src + off, (int32_t*)dst, (uint64_t)n);
            else if (F.src_w == 2 && F.src_unsigned) arrow_widen_kernel<uint16_t, int32_t><<<g, 256, 0, e.copy_stream>>>((const uint16_t*)src + off, (int32_t*)dst, (uint64_t)n);
            else if (F.src_w == 2) arrow_widen_kernel<int16_t, int32_t><<<g, 256, 0, e.copy_stream>>>((const int16_t*)src + off, (int32_t*)dst, (uint64_t)n);
            else arrow_widen_kernel<uint32_t, int64_t><<<g, 256, 0, e.copy_stream>>>((const uint32_t*)src + off, (int64_t*)dst, (uint64_t)n);
            TG_CUDA(cudaGetLastError());
            e.launches += 1;
        } else if (F.src_unsigned && F.src_w == 8) {
            dev_check_aligned(src, 8, "the values of column '" + name + "'");
            arrow_u64_kernel<<<g, 256, 0, e.copy_stream>>>((const uint64_t*)src + off, (uint64_t*)dst, (uint64_t)n, validity, (uint64_t)off, flags);
            TG_CUDA(cudaGetLastError());
            e.launches += 1;
        } else {
            TG_CUDA(cudaMemcpyAsync(dst, src + off * w, (size_t)n * w, cudaMemcpyDefault, e.copy_stream));
        }
        c.value_bytes = (have + n) * (int64_t)w;
        if (dtype == TG_INT64 || dtype == TG_FLOAT64) {
            k.pivot = true;
            k.pivot_bits = validity;
            k.pivot_bit0 = off;
        }
        B.extract_validity(i, validity, off);
    }
    c.n_rows = have + n;
}

void table_append_arrow_device(Table& t, const void* schema_p, const void* device_array_p) {
    const ArrowDeviceArray* da = (const ArrowDeviceArray*)device_array_p;
    if (!da) throw Error(TG_ERR_INVALID_ARG, "expected a struct-typed ArrowDeviceArray (a RecordBatch)");
    Engine& e = *t.eng;
    switch (da->device_type) {
        case ARROW_DEVICE_CPU: return table_append_arrow(t, schema_p, &da->array);
        case ARROW_DEVICE_CUDA_HOST: {
            if (da->sync_event) TG_CUDA(cudaEventSynchronize(*(cudaEvent_t*)da->sync_event));
            table_append_arrow(t, schema_p, &da->array);
            TG_CUDA(cudaStreamSynchronize(e.copy_stream));  // pinned buffers are copied asynchronously: the producer may reuse them on return
            return;
        }
        case ARROW_DEVICE_CUDA:
        case ARROW_DEVICE_CUDA_MANAGED: break;
        default: throw Error(TG_ERR_UNSUPPORTED, "Arrow device type " + std::to_string(da->device_type) + " is not supported (CPU, CUDA, CUDA_HOST, CUDA_MANAGED)");
    }
    const ArrowSchema* sc = (const ArrowSchema*)schema_p;
    const ArrowArray* ar = &da->array;
    if (!sc || !sc->format || strcmp(sc->format, "+s") != 0) throw Error(TG_ERR_INVALID_ARG, "expected a struct-typed ArrowArray (a RecordBatch)");
    if (ar->offset != 0) throw Error(TG_ERR_UNSUPPORTED, "sliced struct arrays are not supported");
    if (da->device_id != e.device)
        throw Error(TG_ERR_INVALID_ARG, "the device array lies on device " + std::to_string(da->device_id) + ", not on the engine's device " + std::to_string(e.device));
    // checked before any copy or kernel: a host pointer labelled CUDA, or another GPU's memory, is refused, not dereferenced
    for (int64_t i = 0; i < sc->n_children; ++i) dev_check_child(e, sc->children[i], ar->children[i]);
    AppendTxn txn(t);  // a child that fails undoes the children before it
    if (da->sync_event) TG_CUDA(cudaStreamWaitEvent(e.copy_stream, *(cudaEvent_t*)da->sync_event, 0));
    DevBatch B{e};
    const size_t nc = (size_t)std::max<int64_t>(sc->n_children, 0);
    B.ch.resize(nc);
    if (nc) {
        const size_t rb = r16(nc * sizeof(ArrowDevResult));
        uint8_t* p = e.dev_alloc(rb);
        e.deferred_free.emplace_back(p, rb);
        TG_CUDA(cudaMemsetAsync(p, 0, rb, e.copy_stream));
        B.d_res = (ArrowDevResult*)p;
    }
    for (size_t i = 0; i < nc; ++i) {
        const ArrowSchema* cs = sc->children[i];
        const ArrowArray* ca = ar->children[i];
        B.ch[i].name = cs->name ? cs->name : "";
        B.ch[i].n = ca->length;
        try {
            if (ca->length < 0 || ca->offset < 0) throw Error(TG_ERR_INVALID_ARG, "column '" + B.ch[i].name + "': negative length or offset");
            const std::string fmt = cs->format;
            if (cs->dictionary) {  // the host path's rules (table_append_arrow)
                const char* vf = cs->dictionary->format;
                const bool int_index = fmt.size() == 1 && strchr("cCsSiIlL", fmt[0]) != nullptr;
                const bool utf8_values = vf && (strcmp(vf, "u") == 0 || strcmp(vf, "U") == 0);
                if (!int_index || !utf8_values || !ca->dictionary)
                    throw Error(TG_ERR_UNSUPPORTED, std::string("column '") + cs->name + "': dictionary of " + arrow_type_name(vf) +
                                                        " values (index type " + arrow_type_name(fmt.c_str()) + ") is not supported; string dictionaries only");
                append_dev_dict_utf8(txn, B, i, fmt[0], vf[0] == 'U', ca, ca->dictionary);
                continue;
            }
            if (fmt == "vu") {
                append_dev_view_utf8(txn, B, i, ca);
                continue;
            }
            if (fmt == "vz") throw Error(TG_ERR_UNSUPPORTED, std::string("column '") + cs->name + "': BinaryView is not supported");
            const ArrowFormat F = arrow_format(fmt, cs->name);
            if (F.src_type) {
                Column* have = t.find(cs->name);
                if (have && (have->src_type == nullptr || strcmp(have->src_type, F.src_type) != 0))
                    throw Error(TG_ERR_TYPE_MISMATCH, std::string("column '") + cs->name + "' was registered with a different type");
            }
            append_dev_plain(txn, B, i, F, ca);
            if (F.src_type) {
                Column* c = B.ch[i].c;
                c->src_type = F.src_type;
                c->src_unsigned = F.src_unsigned;
                c->temporal = F.temporal;
                c->temporal_unit = F.temporal_unit;
            }
        } catch (Error&) {
            B.read_back(i);  // an earlier child's flag is the batch's first error, as on the host path
            throw;
        }
    }
    // the one read-back of the batch: flags, NULL counts and last 64 bits of every child. After it, no copy or kernel that
    // reads the producer's buffers is pending (they were queued before it on copy_stream): the producer may reuse them.
    const std::vector<ArrowDevResult> r = B.read_back(nc);
    // pivots: the first (up to) 65536 new values of a column without one, and their validity, read back together
    std::vector<std::vector<uint8_t>> pv(nc), pb(nc);
    bool any_pivot = false;
    for (size_t i = 0; i < nc; ++i) {
        const DevChild& k = B.ch[i];
        if (!k.pivot || k.c->pivot_set || k.n == 0) continue;
        const int64_t head = std::min<int64_t>(k.n, 65536);
        pv[i].resize((size_t)head * 8);
        dev_read(e, pv[i].data(), k.c->values.p + (size_t)k.have * 8, pv[i].size());
        if (k.pivot_bits) {
            pb[i].resize((size_t)((k.pivot_bit0 & 7) + head + 7) / 8);
            dev_read(e, pb[i].data(), k.pivot_bits + k.pivot_bit0 / 8, pb[i].size());
        }
        any_pivot = true;
    }
    if (any_pivot) TG_CUDA(cudaStreamSynchronize(e.copy_stream));
    for (size_t i = 0; i < nc; ++i) {
        DevChild& k = B.ch[i];
        if (!k.c || k.n == 0) continue;
        Column& c = *k.c;
        if (!pv[i].empty()) set_pivot_host(c, c.dtype, (int64_t)pv[i].size() / 8, pv[i].data(), pb[i].empty() ? nullptr : pb[i].data(), k.pivot_bit0 & 7);
        if (k.vwords) append_validity_device(e, c, k.have, k.vwords, k.n, (int64_t)r[i].zeros, r[i].last64);
        else append_validity(e, c, k.have, nullptr, 0, k.n);
        if (k.bwords) {
            append_bits_device(e, c.values, c.tail_vbyte, k.have, k.bwords, k.n, r[i].vlast64);
            c.value_bytes = (k.have + k.n + 7) / 8;
        }
    }
    txn.commit();
}

}  // namespace tg
