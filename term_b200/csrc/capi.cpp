// extern "C" surface declared in include/termgpu.h
#include <cstring>

#include "arrow_abi.h"
#include "engine.hpp"
#include "hashpart.hpp"
#include "radix_sort.cuh"
#include "regex_dfa.hpp"

namespace tg {
const char* last_error_cstr();
Column* table_get_or_add(Table& t, const std::string& name, int32_t dtype);
void table_append_host(Table& t, const std::string& name, int32_t dtype, int64_t n, const void* values,
                       const int32_t* offsets, const uint8_t* validity, int64_t bit_offset);
void table_append_parquet_chunk(Table& t, const std::string& name, int32_t dtype, int32_t max_def_level, int32_t codec,
                                const uint8_t* chunk, int64_t n_bytes, int64_t num_values);
int32_t parquet_inspect_chunk(const uint8_t* chunk, int64_t n_bytes, tg_parquet_page* pages, int32_t cap);
int64_t parquet_chunk_validity(const uint8_t* chunk, int64_t n_bytes, int64_t num_values, uint8_t* out_bits);
int64_t parquet_snappy_decompress(const uint8_t* src, int64_t n, uint8_t* dst, int64_t cap);
int64_t parquet_page_decompress(int32_t codec, const uint8_t* src, int64_t n, uint8_t* dst, int64_t cap);
void table_set_column_arrow_type(Table& t, const std::string& name, const std::string& fmt);
int64_t parquet_decode_to_plain(int32_t encoding, int32_t elem_width, const uint8_t* src, int64_t n, int64_t n_values, uint8_t* dst, int64_t cap);
void table_adopt_device(Table& t, const std::string& name, int32_t dtype, int64_t n, const void* d_values,
                        const int32_t* d_offsets, const uint8_t* d_validity, int64_t n_value_bytes);
void table_append_arrow(Table& t, const void* schema_p, const void* array_p);
void table_append_arrow_device(Table& t, const void* schema_p, const void* device_array_p);
void table_append_csv(Table& t, const std::vector<std::string>& names, const std::vector<std::string>& fmts, const uint8_t* bytes, int64_t n_bytes,
                      const tg_csv_format* format, int64_t* rows_out);
void csv_parse_value(const std::string& fmt, const uint8_t* p, int64_t n, void* out, int32_t* is_null);
void csv_split_host(const tg_csv_format* format, const uint8_t* p, int64_t n, uint8_t* values, int64_t* value_ends, uint8_t* is_null,
                    int64_t* record_fields, int64_t* record_lines, int64_t* n_fields, int64_t* n_records);
}  // namespace tg

using namespace tg;

struct tg_engine {
    Engine e;
};
struct tg_table {
    Table t;
};
struct tg_plan {
    Plan p;
    std::string msg_scratch;
};

static std::vector<std::string> strvec(const char* const* a, int32_t n) {
    std::vector<std::string> v;
    for (int32_t i = 0; i < n; ++i) v.emplace_back(a[i] ? a[i] : "");
    return v;
}

template <typename F>
static tg_status guard(F&& f) {
    try {
        f();
        return TG_OK;
    } catch (Error& e) {
        return fail(e.code, e.msg);
    } catch (std::exception& e) {
        return fail(TG_ERR_INTERNAL, e.what());
    }
}
template <typename F>
static int32_t guard_slot(F&& f) {
    try {
        return f();
    } catch (Error& e) {
        fail(e.code, e.msg);
        return -(int32_t)e.code;
    } catch (std::exception& e) {
        fail(TG_ERR_INTERNAL, e.what());
        return -(int32_t)TG_ERR_INTERNAL;
    }
}

extern "C" {

const char* tg_last_error(void) { return last_error_cstr(); }
const char* tg_version(void) { return "termgpu 0.1.0 (sm_100a)"; }

tg_status tg_engine_create(int device, tg_engine** out) {
    return guard([&] {
        if (!out) throw Error(TG_ERR_INVALID_ARG, "out is NULL");
        int n = 0;
        cudaError_t ce = cudaGetDeviceCount(&n);
        if (ce != cudaSuccess || n == 0)
            throw Error(TG_ERR_CUDA, std::string("no CUDA device available (termgpu has no CPU fallback): ") +
                                         cudaGetErrorString(ce));
        if (device < 0 || device >= n) throw Error(TG_ERR_INVALID_ARG, "device index out of range");
        TG_CUDA(cudaSetDevice(device));
        auto* h = new tg_engine();
        Engine& e = h->e;
        e.device = device;
        cudaDeviceProp prop{};
        TG_CUDA(cudaGetDeviceProperties(&prop, device));
        e.sm_count = prop.multiProcessorCount;
        TG_CUDA(cudaStreamCreateWithFlags(&e.stream, cudaStreamNonBlocking));
        TG_CUDA(cudaStreamCreateWithFlags(&e.copy_stream, cudaStreamNonBlocking));
        for (auto& ev : e.ev) TG_CUDA(cudaEventCreate(&ev));
        e.pinned_bytes = 32u << 20;
        for (int i = 0; i < 2; ++i) {
            TG_CUDA(cudaMallocHost(&e.pinned[i], e.pinned_bytes));
            TG_CUDA(cudaEventCreateWithFlags(&e.pinned_free[i], cudaEventDisableTiming));
        }
        *out = h;
    });
}

void tg_engine_destroy(tg_engine* h) {
    if (!h) return;
    Engine& e = h->e;
    cudaSetDevice(e.device);
    cudaDeviceSynchronize();
    rank_session_destroy(e);
    try {
        comm_destroy(e);
    } catch (...) {
    }
    for (auto& kv : e.tables) {
        for (auto& c : kv.second->cols) {
            if (c->values.owned && c->values.p) cudaFree(c->values.p);
            if (c->offsets.owned && c->offsets.p) cudaFree(c->offsets.p);
            if (c->validity.owned && c->validity.p) cudaFree(c->validity.p);
            if (c->wide && c->wide->values.owned && c->wide->values.p) cudaFree(c->wide->values.p);
        }
    }
    e.tables.clear();
    {
        std::lock_guard<std::mutex> g(e.mask_returns->mu);
        for (auto& b : e.mask_returns->blocks) cudaFree(b.first);
        e.mask_returns->blocks.clear();
        e.mask_returns->engine_alive = false;
    }
    for (auto& b : e.deferred_free) cudaFree(b.first);  // the device is idle (synchronised above)
    e.deferred_free.clear();
    e.dev_trim();
    if (e.d_scratch) cudaFree(e.d_scratch);
    if (e.d_shuffle) cudaFree(e.d_shuffle);
    if (e.d_aux) cudaFree(e.d_aux);
    mailbox_destroy(e);
    for (auto& s : e.side)
        if (s) cudaStreamDestroy(s);
    for (auto& ev : e.side_ev)
        if (ev) cudaEventDestroy(ev);
    if (e.h_scratch) cudaFreeHost(e.h_scratch);
    for (int i = 0; i < 2; ++i) {
        if (e.pinned[i]) cudaFreeHost(e.pinned[i]);
        if (e.pinned_free[i]) cudaEventDestroy(e.pinned_free[i]);
    }
    for (auto& ev : e.ev)
        if (ev) cudaEventDestroy(ev);
    if (e.stream) cudaStreamDestroy(e.stream);
    if (e.copy_stream) cudaStreamDestroy(e.copy_stream);
    delete h;
}

uint64_t tg_engine_launch_count(const tg_engine* h) { return h ? h->e.launches : 0; }
void* tg_engine_stream(tg_engine* h) { return h ? (void*)h->e.stream : nullptr; }

// tables are owned by the engine's registry; tg_table* is a borrowed handle
tg_status tg_engine_sync_copies(tg_engine* h) {
    return guard([&] {
        if (!h) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        std::lock_guard<std::mutex> g(h->e.mu);
        TG_CUDA(cudaSetDevice(h->e.device));
        h->e.sync_copies();
    });
}

tg_status tg_table_create(tg_engine* h, const char* name, tg_table** out) {
    return guard([&] {
        if (!h || !name || !out) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        validate_identifier(name);
        std::lock_guard<std::mutex> g(h->e.mu);
        if (h->e.tables.count(name)) throw Error(TG_ERR_INVALID_ARG, std::string("table '") + name + "' already exists");
        auto t = std::make_unique<Table>();
        t->eng = &h->e;
        t->name = name;
        Table* raw = t.get();
        h->e.tables[name] = std::move(t);
        *out = reinterpret_cast<tg_table*>(raw);
    });
}

tg_status tg_table_drop(tg_engine* h, const char* name) {
    return guard([&] {
        if (!h || !name) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        std::lock_guard<std::mutex> g(h->e.mu);
        auto it = h->e.tables.find(name);
        if (it == h->e.tables.end()) throw Error(TG_ERR_TABLE_NOT_FOUND, std::string("table '") + name + "' not found");
        cudaSetDevice(h->e.device);
        cudaStreamSynchronize(h->e.copy_stream);
        cudaStreamSynchronize(h->e.stream);
        for (auto& c : it->second->cols) column_free(h->e, *c);
        h->e.tables.erase(it);
    });
}

tg_status tg_table_partition_fingerprints(tg_engine* h, const char* table, const char* const* columns, int32_t n_columns, int32_t n_parts,
                                          void** d_records, int64_t* counts) {
    return guard([&] {
        if (!h || !table || !columns || !d_records || !counts) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        Engine& e = h->e;
        std::lock_guard<std::mutex> g(e.mu);
        TG_CUDA(cudaSetDevice(e.device));
        e.sync_copies();
        auto it = e.tables.find(table);
        if (it == e.tables.end()) throw Error(TG_ERR_TABLE_NOT_FOUND, std::string("table '") + table + "' not found");
        int launches = 0;
        partition_fingerprints_by_rank(e, *it->second, strvec(columns, n_columns), n_parts, d_records, counts, launches);
        e.launches += launches;
    });
}

tg_status tg_table_column_dtype(const tg_table* t, const char* column, int32_t* dtype) {
    return guard([&] {
        if (!t || !column || !dtype) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        Table* tab = const_cast<Table*>(reinterpret_cast<const Table*>(t));
        Column* c = tab->find(column);
        if (!c) throw Error(TG_ERR_COLUMN_NOT_FOUND, "Schema error: No field named " + std::string(column) + ". Valid fields are " + tab->valid_fields() + ".");
        *dtype = c->dtype;
    });
}

tg_status tg_table_column_buffers(tg_engine* h, const char* table, const char* column, tg_column_buffers* out) {
    return guard([&] {
        if (!h || !table || !column || !out) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        Engine& e = h->e;
        std::lock_guard<std::mutex> g(e.mu);
        auto it = e.tables.find(table);
        if (it == e.tables.end())
            throw Error(TG_ERR_TABLE_NOT_FOUND, "Error during planning: table 'datafusion.public." + std::string(table) + "' not found");
        Column* c = it->second->find(column);
        if (!c) throw Error(TG_ERR_COLUMN_NOT_FOUND, "Schema error: No field named " + std::string(column) + ". Valid fields are " + it->second->valid_fields() + ".");
        e.sync_copies();
        *out = tg_column_buffers{c->dtype, it->second->n_rows, c->values.p, c->offsets.p, c->validity.p, c->value_bytes, c->null_count};
    });
}

tg_status tg_table_partition_keys(tg_engine* h, const char* table, const char* column, int32_t n_parts, void** d_keys,
                                  int64_t* counts, int64_t* n_null_rows) {
    return guard([&] {
        if (!h || !table || !column || !d_keys || !counts || !n_null_rows) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        Engine& e = h->e;
        std::lock_guard<std::mutex> g(e.mu);
        TG_CUDA(cudaSetDevice(e.device));
        e.sync_copies();
        auto it = e.tables.find(table);
        if (it == e.tables.end()) throw Error(TG_ERR_TABLE_NOT_FOUND, std::string("table '") + table + "' not found");
        Table& t = *it->second;
        Column* c = t.find(column);
        if (!c) throw Error(TG_ERR_COLUMN_NOT_FOUND, "Schema error: No field named " + std::string(column) + ". Valid fields are " + t.valid_fields() + ".");
        c = numeric_view(e, c);  // (Int32 / Float32 keys travel as their exactly widened values)
        if (!c) throw Error(TG_ERR_TYPE_MISMATCH, "the multi-GPU key shuffle supports numeric key columns (strings travel as fingerprints)");
        uint64_t* keys = nullptr;
        int launches = 0;
        partition_keys_by_rank(e, *c, t.n_rows, n_parts, &keys, counts, n_null_rows, launches);
        e.launches += launches;
        *d_keys = keys;
    });
}

tg_status tg_table_lookup(tg_engine* h, const char* name, tg_table** out) {
    return guard([&] {
        if (!h || !name || !out) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        std::lock_guard<std::mutex> g(h->e.mu);
        auto it = h->e.tables.find(name);
        if (it == h->e.tables.end()) throw Error(TG_ERR_TABLE_NOT_FOUND, std::string("table '") + name + "' not found");
        *out = reinterpret_cast<tg_table*>(it->second.get());
    });
}

int64_t tg_table_num_rows(const tg_table* t) { return t ? reinterpret_cast<const Table*>(t)->n_rows : -1; }

tg_status tg_table_append_host(tg_table* t, const char* name, int32_t dtype, int64_t n_rows, const void* values,
                               const int32_t* offsets, const uint8_t* validity, int64_t bit_offset) {
    return guard([&] {
        if (!t || !name) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        table_append_host(*reinterpret_cast<Table*>(t), name, dtype, n_rows, values, offsets, validity, bit_offset);
    });
}

tg_status tg_table_append_parquet_chunk(tg_table* t, const char* name, int32_t dtype, int32_t max_definition_level, int32_t codec,
                                        const void* chunk, int64_t n_bytes, int64_t num_values) {
    return guard([&] {
        if (!t || !name) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        table_append_parquet_chunk(*reinterpret_cast<Table*>(t), name, dtype, max_definition_level, codec, (const uint8_t*)chunk, n_bytes,
                                   num_values);
    });
}
int64_t tg_parquet_chunk_validity(const void* chunk, int64_t n_bytes, int64_t num_values, uint8_t* out_bits) {
    int64_t n = 0;
    tg_status st = guard([&] { n = parquet_chunk_validity((const uint8_t*)chunk, n_bytes, num_values, out_bits); });
    return st == TG_OK ? n : -(int64_t)st;
}
int64_t tg_parquet_snappy_decompress(const void* src, int64_t n_bytes, void* dst, int64_t cap) {
    int64_t n = 0;
    tg_status st = guard([&] { n = parquet_snappy_decompress((const uint8_t*)src, n_bytes, (uint8_t*)dst, cap); });
    return st == TG_OK ? n : -(int64_t)st;
}
tg_status tg_table_set_column_arrow_type(tg_table* t, const char* column, const char* arrow_format) {
    return guard([&] {
        if (!t || !column || !arrow_format) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        table_set_column_arrow_type(*reinterpret_cast<Table*>(t), column, arrow_format);
    });
}
int64_t tg_parquet_decode_to_plain(int32_t encoding, int32_t elem_width, const void* src, int64_t n_bytes, int64_t n_values, void* dst, int64_t cap) {
    int64_t n = 0;
    tg_status st = guard([&] { n = parquet_decode_to_plain(encoding, elem_width, (const uint8_t*)src, n_bytes, n_values, (uint8_t*)dst, cap); });
    return st == TG_OK ? n : -(int64_t)st;
}
int64_t tg_parquet_page_decompress(int32_t codec, const void* src, int64_t n_bytes, void* dst, int64_t cap) {
    int64_t n = 0;
    tg_status st = guard([&] { n = parquet_page_decompress(codec, (const uint8_t*)src, n_bytes, (uint8_t*)dst, cap); });
    return st == TG_OK ? n : -(int64_t)st;
}
int32_t tg_parquet_inspect_chunk(const void* chunk, int64_t n_bytes, tg_parquet_page* pages, int32_t cap) {
    int32_t n = 0;
    tg_status st = guard([&] { n = parquet_inspect_chunk((const uint8_t*)chunk, n_bytes, pages, cap); });
    return st == TG_OK ? n : -(int32_t)st;
}

tg_status tg_table_adopt_device(tg_table* t, const char* name, int32_t dtype, int64_t n_rows, const void* d_values,
                                const int32_t* d_offsets, const uint8_t* d_validity, int64_t n_value_bytes) {
    return guard([&] {
        if (!t || !name) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        table_adopt_device(*reinterpret_cast<Table*>(t), name, dtype, n_rows, d_values, d_offsets, d_validity,
                           n_value_bytes);
    });
}

tg_status tg_table_append_csv(tg_table* t, const char* const* columns, const char* const* arrow_formats, int32_t n_columns, const void* bytes,
                              int64_t n_bytes, int32_t delimiter, int32_t has_header, int64_t* rows_out) {
    if (delimiter < 0 || delimiter > 255) return fail(TG_ERR_INVALID_ARG, "CSV: the delimiter must be a byte (0..255)");
    const tg_csv_format f{delimiter, -1, -1, -1, -1, has_header, nullptr};
    return tg_table_append_csv_format(t, columns, arrow_formats, n_columns, bytes, n_bytes, &f, rows_out);
}
tg_status tg_table_append_csv_format(tg_table* t, const char* const* columns, const char* const* arrow_formats, int32_t n_columns, const void* bytes,
                                     int64_t n_bytes, const tg_csv_format* format, int64_t* rows_out) {
    return guard([&] {
        if (!t || (n_columns > 0 && (!columns || !arrow_formats)) || n_columns < 0) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        std::vector<std::string> names, fmts;
        for (int32_t i = 0; i < n_columns; ++i) {
            if (!columns[i] || !arrow_formats[i]) throw Error(TG_ERR_INVALID_ARG, "NULL column name or format");
            names.emplace_back(columns[i]);
            fmts.emplace_back(arrow_formats[i]);
        }
        table_append_csv(*reinterpret_cast<Table*>(t), names, fmts, (const uint8_t*)bytes, n_bytes, format, rows_out);
    });
}
tg_status tg_csv_split_host(const tg_csv_format* format, const void* bytes, int64_t n_bytes, uint8_t* values, int64_t* value_ends, uint8_t* is_null,
                            int64_t* record_fields, int64_t* record_lines, int64_t* n_fields, int64_t* n_records) {
    return guard([&] {
        csv_split_host(format, (const uint8_t*)bytes, n_bytes, values, value_ends, is_null, record_fields, record_lines, n_fields, n_records);
    });
}
tg_status tg_csv_parse_value(const char* arrow_format, const void* field, int64_t n_bytes, void* out, int32_t* is_null) {
    return guard([&] {
        if (!arrow_format) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        csv_parse_value(arrow_format, (const uint8_t*)field, n_bytes, out, is_null);
    });
}
tg_status tg_table_append_arrow(tg_table* t, const void* schema, const void* array) {
    return guard([&] {
        if (!t) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        table_append_arrow(*reinterpret_cast<Table*>(t), schema, array);
    });
}
tg_status tg_table_append_arrow_device(tg_table* t, const void* schema, const void* device_array) {
    return guard([&] {
        if (!t) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        table_append_arrow_device(*reinterpret_cast<Table*>(t), schema, device_array);
    });
}

// ------------------------------------------------------------------ plan ----
tg_status tg_plan_create(tg_plan** out) {
    return guard([&] {
        if (!out) throw Error(TG_ERR_INVALID_ARG, "out is NULL");
        *out = new tg_plan();
    });
}
void tg_plan_destroy(tg_plan* p) { delete p; }
int32_t tg_plan_num_slots(const tg_plan* p) { return p ? (int32_t)p->p.slots.size() : 0; }


int32_t tg_plan_add_completeness(tg_plan* p, const char* const* columns, int32_t n, double threshold, int32_t op,
                                 int32_t op_n) {
    return guard_slot([&] { return plan_add_completeness(p->p, strvec(columns, n), threshold, op, op_n); });
}
int32_t tg_plan_add_size(tg_plan* p, tg_assertion a) {
    return guard_slot([&] { return plan_add_size(p->p, a); });
}
int32_t tg_plan_add_statistic(tg_plan* p, const char* column, int32_t kind, double pct, tg_assertion a) {
    return guard_slot([&] { return plan_add_statistic(p->p, column ? column : "", kind, pct, a); });
}
int32_t tg_plan_add_multi_statistic(tg_plan* p, const char* column, const int32_t* kinds, const double* pcts,
                                    const tg_assertion* as, int32_t n) {
    return guard_slot([&] {
        std::vector<StatReq> v;
        for (int32_t i = 0; i < n; ++i) v.push_back(StatReq{kinds[i], pcts ? pcts[i] : 0.0, as[i], -1});
        return plan_add_multi_statistic(p->p, column ? column : "", v);
    });
}
int32_t tg_plan_add_format(tg_plan* p, const char* column, int32_t kind, const char* arg, int32_t flag,
                           double threshold, const tg_format_options* opt) {
    return guard_slot([&] {
        tg_format_options o{1, 0, 1};
        if (opt) o = *opt;
        return plan_add_format(p->p, column ? column : "", kind, arg, flag, threshold, o);
    });
}
int32_t tg_plan_add_uniqueness(tg_plan* p, const char* const* columns, int32_t n, int32_t kind, double threshold,
                               tg_assertion a, int32_t null_handling) {
    return guard_slot([&] { return plan_add_uniqueness(p->p, strvec(columns, n), kind, threshold, a, null_handling); });
}
int32_t tg_plan_add_correlation(tg_plan* p, const char* c1, const char* c2, int32_t kind, tg_assertion a) {
    return guard_slot([&] { return plan_add_correlation(p->p, c1 ? c1 : "", c2 ? c2 : "", kind, a); });
}
int32_t tg_plan_add_custom_sql(tg_plan* p, const char* expr, const char* hint) {
    return guard_slot([&] { return plan_add_custom_sql(p->p, expr ? expr : "", hint); });
}
int32_t tg_plan_add_foreign_key(tg_plan* p, const char* child, const char* parent, int32_t allow_nulls,
                                int32_t max_examples) {
    return guard_slot([&] { return plan_add_foreign_key(p->p, child ? child : "", parent ? parent : "", allow_nulls, max_examples); });
}
int32_t tg_plan_add_analyzer(tg_plan* p, int32_t kind, const char* column, const char* column2, const char* expr) {
    return guard_slot([&] { return plan_add_analyzer(p->p, kind, column, column2, expr); });
}
int32_t tg_plan_add_kll(tg_plan* p, const char* column, int32_t k, const double* q, int32_t nq) {
    return guard_slot([&] {
        std::vector<double> v(q, q + (nq > 0 ? nq : 0));
        return plan_add_kll(p->p, column ? column : "", k, v);
    });
}
int32_t tg_plan_add_length(tg_plan* p, const char* column, int32_t kind, int64_t a, int64_t b) {
    return guard_slot([&] { return plan_add_length(p->p, column ? column : "", kind, a, b); });
}
int32_t tg_plan_add_containment(tg_plan* p, const char* column, const char* const* allowed, int32_t n) {
    return guard_slot([&] { return plan_add_containment(p->p, column ? column : "", strvec(allowed, n)); });
}
int32_t tg_plan_add_non_negative(tg_plan* p, const char* column) {
    return guard_slot([&] { return plan_add_non_negative(p->p, column ? column : ""); });
}
int32_t tg_plan_add_approx_count_distinct(tg_plan* p, const char* column, tg_assertion a) {
    return guard_slot([&] { return plan_add_approx_count_distinct(p->p, column ? column : "", a); });
}
int32_t tg_plan_add_data_type(tg_plan* p, const char* column, int32_t data_type, double threshold) {
    return guard_slot([&] { return plan_add_data_type(p->p, column ? column : "", data_type, threshold); });
}
int32_t tg_plan_add_column_count(tg_plan* p, tg_assertion a) {
    return guard_slot([&] { return plan_add_column_count(p->p, a); });
}
int32_t tg_plan_add_quantile(tg_plan* p, const char* column, int32_t validation, const double* quantiles,
                             const tg_assertion* assertions, int32_t n, int32_t strict) {
    return guard_slot([&] {
        std::vector<double> q;
        std::vector<tg_assertion> a;
        for (int32_t i = 0; i < n; ++i) {
            q.push_back(quantiles[i]);
            if (assertions) a.push_back(assertions[i]);
        }
        return plan_add_quantile(p->p, column ? column : "", validation, q, a, strict);
    });
}
int32_t tg_plan_add_histogram(tg_plan* p, const char* column, int32_t num_buckets) {
    return guard_slot([&] { return plan_add_histogram(p->p, column ? column : "", num_buckets); });
}
int32_t tg_plan_add_value_histogram(tg_plan* p, const char* column) {
    return guard_slot([&] { return plan_add_value_histogram(p->p, column ? column : ""); });
}
int32_t tg_plan_add_grouped_completeness(tg_plan* p, const char* column, const char* const* groups, int32_t n,
                                         int32_t max_groups, int32_t include_overall) {
    return guard_slot([&] {
        return plan_add_grouped_completeness(p->p, column ? column : "", strvec(groups, n), max_groups, include_overall);
    });
}

tg_status tg_plan_execute_partial(tg_engine* h, tg_plan* p, const char* table_name) {
    return guard([&] {
        if (!h || !p) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        execute_partial(h->e, p->p, table_name ? table_name : "data");
    });
}
tg_status tg_plan_execute(tg_engine* h, tg_plan* p, const char* table_name) {
    return guard([&] {
        if (!h || !p) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        execute_partial(h->e, p->p, table_name ? table_name : "data");
        p->p.finalize();
    });
}
tg_status tg_plan_request_row_mask(tg_plan* p, int32_t slot) {
    return guard([&] {
        if (!p) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        plan_request_row_mask(p->p, slot);
    });
}

// private data of an exported row mask: the schema owns nothing; the array keeps the mask's buffers alive
struct RowMaskExport {
    std::shared_ptr<RowMask> mask;
    const void* buffers[2];
};
static void row_mask_release_schema(ArrowSchema* s) { s->release = nullptr; }
static void row_mask_release_array(ArrowArray* a) {
    delete static_cast<RowMaskExport*>(a->private_data);
    a->release = nullptr;
}

// fills the Arrow structs of one verdict array; the array shares ownership of the buffers with the slot
static void export_mask(const std::shared_ptr<RowMask>& mask, void* arrow_schema_out, void* arrow_device_array_out) {
    const RowMask& m = *mask;
    auto* x = new RowMaskExport{mask, {m.validity, m.values}};
    ArrowSchema* sc = static_cast<ArrowSchema*>(arrow_schema_out);
    *sc = ArrowSchema{};
    sc->format = "b";
    sc->name = "";
    sc->flags = 2;  // ARROW_FLAG_NULLABLE
    sc->release = row_mask_release_schema;
    ArrowDeviceArray* da = static_cast<ArrowDeviceArray*>(arrow_device_array_out);
    *da = ArrowDeviceArray{};
    da->array.length = m.n_rows;
    da->array.null_count = m.null_count;
    da->array.n_buffers = 2;
    da->array.buffers = x->buffers;
    da->array.release = row_mask_release_array;
    da->array.private_data = x;
    da->device_id = m.device;
    da->device_type = ARROW_DEVICE_CUDA;
    da->sync_event = nullptr;
}

tg_status tg_plan_export_row_mask(const tg_plan* p, int32_t slot, void* arrow_schema_out, void* arrow_device_array_out) {
    return guard([&] {
        if (!p || !arrow_schema_out || !arrow_device_array_out) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        if (slot < 0 || slot >= (int32_t)p->p.slots.size()) throw Error(TG_ERR_INVALID_ARG, "slot index out of range");
        const Slot& s = p->p.slots[slot];
        if (!s.mask_requested) throw Error(TG_ERR_INVALID_ARG, "row mask of slot " + std::to_string(slot) + " was not requested");
        if (!s.mask_built) throw Error(TG_ERR_INVALID_ARG, "row mask of slot " + std::to_string(slot) + " was requested but the plan was not executed since");
        if (s.mask_err != TG_OK) throw Error(s.mask_err, s.mask_err_msg);
        export_mask(s.mask, arrow_schema_out, arrow_device_array_out);
    });
}

tg_status tg_plan_request_key_rows(tg_plan* p, int32_t slot, int32_t kind) {
    return guard([&] {
        if (!p) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        plan_request_key_rows(p->p, slot, kind);
    });
}

tg_status tg_plan_export_key_rows(const tg_plan* p, int32_t slot, int32_t kind, void* arrow_schema_out, void* arrow_device_array_out) {
    return guard([&] {
        if (!p || !arrow_schema_out || !arrow_device_array_out) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        const Slot& s = key_rows_slot(p->p, slot, kind);
        const std::string what = "key-level row verdicts (kind " + std::to_string(kind) + ") of slot " + std::to_string(slot);
        if (!(s.key_rows_requested & (1u << kind))) throw Error(TG_ERR_INVALID_ARG, what + " were not requested");
        if (!s.mask_built) throw Error(TG_ERR_INVALID_ARG, what + " were requested but the plan was not executed since");
        if (s.mask_err != TG_OK) throw Error(s.mask_err, s.mask_err_msg);
        export_mask(s.key_rows[kind], arrow_schema_out, arrow_device_array_out);
    });
}

tg_status tg_plan_partial_size(const tg_plan* p, size_t* n) {
    return guard([&] {
        if (!p || !n) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        *n = p->p.partial_size();
    });
}
tg_status tg_plan_partial_export(const tg_plan* p, void* buf, size_t n) {
    return guard([&] {
        if (!p || !buf) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        if (n < p->p.partial_size()) throw Error(TG_ERR_INVALID_ARG, "buffer too small");
        p->p.partial_export((uint8_t*)buf);
    });
}
tg_status tg_plan_partial_reset(tg_plan* p) {
    return guard([&] {
        if (!p) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        p->p.reset_partials();
    });
}
tg_status tg_plan_partial_merge(tg_plan* p, const void* buf, size_t n) {
    return guard([&] {
        if (!p || !buf) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        p->p.partial_merge((const uint8_t*)buf, n);
    });
}
tg_status tg_plan_finalize(tg_plan* p) {
    return guard([&] {
        if (!p) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        p->p.finalize();
    });
}

int32_t tg_plan_num_aggregates(const tg_plan* p) { return p ? (int32_t)p->p.aggs.size() : 0; }
tg_status tg_plan_aggregate_info(const tg_plan* p, int32_t i, int32_t* kind, const char** key) {
    return guard([&] {
        if (!p || i < 0 || i >= (int32_t)p->p.aggs.size()) throw Error(TG_ERR_INVALID_ARG, "aggregate index out of range");
        if (kind) *kind = p->p.aggs[i].kind;
        if (key) *key = p->p.aggs[i].key.c_str();
    });
}

tg_status tg_engine_mailbox_create(tg_engine* h, int32_t world, int32_t rank, size_t slot_bytes, void* handle_out) {
    return guard([&] {
        if (!h || !handle_out) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        std::lock_guard<std::mutex> g(h->e.mu);
        TG_CUDA(cudaSetDevice(h->e.device));
        mailbox_create(h->e, world, rank, slot_bytes, handle_out);
    });
}
tg_status tg_engine_mailbox_open(tg_engine* h, const void* handles) {
    return guard([&] {
        if (!h || !handles) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        std::lock_guard<std::mutex> g(h->e.mu);
        TG_CUDA(cudaSetDevice(h->e.device));
        mailbox_open(h->e, handles);
    });
}
// publish this plan's partial states to every rank's mailbox, collect everyone's, merge IN RANK ORDER, finalize
tg_status tg_plan_exchange_and_finalize(tg_engine* h, tg_plan* p) {
    return guard([&] {
        if (!h || !p) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        std::vector<uint8_t> blob(p->p.partial_size());
        p->p.partial_export(blob.data());
        std::vector<std::vector<uint8_t>> all;
        if (!mailbox_exchange(h->e, blob.data(), blob.size(), all))
            throw Error(TG_ERR_INVALID_ARG, "mailbox: a rank's partial blob is larger than the slot (use tg_plan_exchange_ex, which reports it)");
        p->p.reset_partials();
        for (auto& b : all) p->p.partial_merge(b.data(), b.size());
        p->p.finalize();
    });
}

// test hook: the hand-written radix sort on its own (host keys -> device -> sort by bits [begin_bit, begin_bit + 8 *
// n_passes) with synthesised row ids -> host)
tg_status tg_debug_sort_pairs(tg_engine* h, const uint64_t* keys, int64_t n, int32_t begin_bit, int32_t n_passes, uint64_t* out_keys,
                              uint32_t* out_index) {
    return guard([&] {
        if (!h || (n > 0 && (!keys || !out_keys || !out_index))) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        if (n < 0 || n >= ((int64_t)1 << 30) || begin_bit < 0 || n_passes < 1 || n_passes > RS_MAX_PASSES || begin_bit + 8 * n_passes > 64)
            throw Error(TG_ERR_INVALID_ARG, "sort range out of bounds");
        if (n == 0) return;
        Engine& e = h->e;
        std::lock_guard<std::mutex> g(e.mu);
        TG_CUDA(cudaSetDevice(e.device));
        const size_t k_b = ((size_t)n * 8 + 255) & ~(size_t)255, i_b = ((size_t)n * 4 + 255) & ~(size_t)255;
        const size_t tmp_b = rs_temp_bytes(n, n_passes);
        uint8_t* scr = e.scratch(2 * k_b + 2 * i_b + tmp_b + 256);
        uint64_t* kb[2] = {(uint64_t*)scr, (uint64_t*)(scr + k_b)};
        uint32_t* vb[2] = {(uint32_t*)(scr + 2 * k_b), (uint32_t*)(scr + 2 * k_b + i_b)};
        const RsTemp T = rs_temp_carve(scr + 2 * k_b + 2 * i_b, n, n_passes);
        TG_CUDA(cudaMemcpyAsync(kb[0], keys, (size_t)n * 8, cudaMemcpyHostToDevice, e.stream));
        const int launches = rs_sort_pairs<uint32_t>(e.stream, kb, vb, n, begin_bit, n_passes, true, T, e.sm_count);
        TG_CUDA(cudaGetLastError());
        e.launches += launches;
        RsControl ctl;
        TG_CUDA(cudaMemcpyAsync(&ctl, T.ctl, sizeof(ctl), cudaMemcpyDeviceToHost, e.stream));
        TG_CUDA(cudaStreamSynchronize(e.stream));
        TG_CUDA(cudaMemcpy(out_keys, kb[ctl.result], (size_t)n * 8, cudaMemcpyDeviceToHost));
        TG_CUDA(cudaMemcpy(out_index, vb[ctl.result], (size_t)n * 4, cudaMemcpyDeviceToHost));
    });
}

// ---- NCCL behind the C ABI (comm.cpp)
tg_status tg_comm_unique_id(void* id128) {
    return guard([&] {
        if (!id128) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        comm_unique_id(id128);
    });
}
tg_status tg_comm_init(tg_engine* h, const void* id128, int32_t world, int32_t rank) {
    return guard([&] {
        if (!h || !id128) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        comm_init(h->e, id128, world, rank);
    });
}
tg_status tg_comm_destroy(tg_engine* h) {
    return guard([&] {
        if (!h) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        std::lock_guard<std::mutex> g(h->e.mu);
        cudaSetDevice(h->e.device);
        comm_destroy(h->e);
    });
}
uint64_t tg_comm_bytes_sent(const tg_engine* h) { return h ? h->e.comm_bytes_sent : 0; }
tg_status tg_table_shuffle_column(tg_engine* h, const char* table, const char* column, const char* shard_table, int32_t partition, int64_t* n_rows) {
    return guard([&] {
        if (!h || !table || !column || !shard_table) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        validate_identifier(shard_table);
        const int64_t n = comm_shuffle_column(h->e, table, column, shard_table, partition == 1);
        if (n_rows) *n_rows = n;
    });
}
tg_status tg_table_shuffle_fingerprints(tg_engine* h, const char* table, const char* const* columns, int32_t n_columns, const char* shard_table,
                                        int64_t* n_rows) {
    return guard([&] {
        if (!h || !table || !columns || n_columns < 1 || !shard_table) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        validate_identifier(shard_table);
        const int64_t n = comm_shuffle_fingerprints(h->e, table, strvec(columns, n_columns), shard_table);
        if (n_rows) *n_rows = n;
    });
}

// ---- distributed RANK() for Spearman (SURVEY §8e K6): the stages of ranks.cu as the host layer's sample sort sees them
tg_status tg_rank_begin(tg_engine* h, const char* table, const char* column_x, const char* column_y, int64_t* n_pairs) {
    return guard([&] {
        if (!h || !table || !column_x || !column_y || !n_pairs) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        *n_pairs = rank_begin(h->e, table, column_x, column_y);
    });
}
tg_status tg_rank_local_sort(tg_engine* h) {
    return guard([&] {
        if (!h) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        rank_local_sort(h->e);
    });
}
int32_t tg_rank_sample(tg_engine* h, int32_t n_samples, uint64_t* keys) {
    return guard_slot([&] {
        if (!h || !keys) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        return rank_sample(h->e, n_samples, keys);
    });
}
tg_status tg_rank_split(tg_engine* h, const uint64_t* splitters, int32_t n_parts, int64_t* counts) {
    return guard([&] {
        if (!h || !counts || (n_parts > 1 && !splitters)) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        rank_split(h->e, splitters, n_parts, counts);
    });
}
tg_status tg_rank_send_buffers(tg_engine* h, const void** keys, const void** payload, int32_t* payload_bytes) {
    return guard([&] {
        if (!h || !keys || !payload || !payload_bytes) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        rank_send_buffers(h->e, keys, payload, payload_bytes);
    });
}
tg_status tg_rank_recv_buffers(tg_engine* h, int64_t n_recv, void** keys, void** payload) {
    return guard([&] {
        if (!h || !keys || !payload) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        rank_recv_buffers(h->e, n_recv, keys, payload);
    });
}
tg_status tg_rank_recv_commit(tg_engine* h, int64_t n_recv) {
    return guard([&] {
        if (!h) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        rank_recv_commit(h->e, n_recv);
    });
}
tg_status tg_rank_finish_x(tg_engine* h, uint64_t rank_base) {
    return guard([&] {
        if (!h) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        rank_finish_x(h->e, rank_base);
    });
}
tg_status tg_rank_finish_y(tg_engine* h, uint64_t rank_base, double center, uint64_t* n_out, double* sums5) {
    return guard([&] {
        if (!h || !n_out || !sums5) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        rank_finish_y(h->e, rank_base, center, n_out, sums5);
    });
}
tg_status tg_rank_exchange(tg_engine* h, int64_t* n_recv, uint64_t* rank_base, uint64_t* total, int32_t* done) {
    return guard([&] {
        if (!h || !n_recv || !rank_base || !total || !done) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        *done = comm_rank_exchange(h->e, n_recv, rank_base, total) ? 1 : 0;
    });
}
tg_status tg_rank_abort(tg_engine* h) {
    return guard([&] {
        if (!h) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        rank_abort(h->e);
    });
}
// a partial state computed outside tg_plan_execute_partial (the distributed rank computation): replaces aggregate i's state
tg_status tg_plan_set_aggregate_partial(tg_plan* p, int32_t i, const uint64_t* u8, const double* f8) {
    return guard([&] {
        if (!p || !u8 || !f8 || i < 0 || i >= (int32_t)p->p.aggs.size()) throw Error(TG_ERR_INVALID_ARG, "aggregate index out of range");
        Agg& a = p->p.aggs[i];
        if (a.kind != A_SPEARMAN) throw Error(TG_ERR_INVALID_ARG, "only SPEARMAN aggregates take an externally computed partial state");
        for (int k = 0; k < 8; ++k) {
            a.u[k] = u8[k];
            a.f[k] = f8[k];
        }
    });
}

// like tg_plan_exchange_and_finalize, but a blob that does not fit some rank's slot is not an error: *fell_back = 1 on
// EVERY rank (the marker travels through the mailbox) and nothing was merged — the host layer then exchanges over NCCL
tg_status tg_plan_exchange_ex(tg_engine* h, tg_plan* p, int32_t* fell_back) {
    return guard([&] {
        if (!h || !p || !fell_back) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        std::vector<uint8_t> blob(p->p.partial_size());
        p->p.partial_export(blob.data());
        std::vector<std::vector<uint8_t>> all;
        *fell_back = mailbox_exchange(h->e, blob.data(), blob.size(), all) ? 0 : 1;
        if (*fell_back) return;
        p->p.reset_partials();
        for (auto& b : all) p->p.partial_merge(b.data(), b.size());
        p->p.finalize();
    });
}
// scan-only plans: partial execute, device-side assembly of the partial states, publish / collect over the peer mailboxes
// and the rank-ordered merge in ONE call with one stream synchronisation. *done = 0: the plan (or the platform) does not
// qualify and nothing was executed — use tg_plan_execute_partial + tg_plan_exchange_ex.
tg_status tg_plan_execute_exchange(tg_engine* h, tg_plan* p, const char* table_name, int32_t* done) {
    return guard([&] {
        if (!h || !p || !table_name || !done) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        *done = execute_exchange_fused(h->e, p->p, table_name) ? 1 : 0;
    });
}

int32_t tg_plan_kll_levels(const tg_plan* p, int32_t slot, int32_t level, double* items, int32_t cap) {
    return guard_slot([&] {
        if (!p) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        if (slot < 0 || slot >= (int32_t)p->p.slots.size()) throw Error(TG_ERR_INVALID_ARG, "slot out of range");
        const Slot& s = p->p.slots[slot];
        int agg = -1;
        for (int a : s.aggs)
            if (p->p.aggs[a].kind == A_KLL) agg = a;
        for (auto& r : s.stats)
            if (r.agg_kll >= 0) agg = r.agg_kll;
        if (agg < 0) throw Error(TG_ERR_INVALID_ARG, "slot has no quantile sketch");
        std::vector<std::vector<double>> levels;
        const int nl = kll_blob_levels(p->p.aggs[agg].blob, levels, nullptr);
        if (nl < 0) return 0;
        if (level < 0) return nl;
        if (level >= nl) return 0;
        const auto& l = levels[level];
        for (size_t i = 0; items && i < l.size() && (int32_t)i < cap; ++i) items[i] = l[i];
        return (int32_t)l.size();
    });
}

int32_t tg_plan_histogram_pending(const tg_plan* p, int32_t* agg_indices, int32_t cap) {
    return guard_slot([&] {
        if (!p) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        const std::vector<int> v = p->p.histogram_pending();
        for (size_t i = 0; agg_indices && i < v.size() && (int32_t)i < cap; ++i) agg_indices[i] = v[i];
        return (int32_t)v.size();
    });
}
tg_status tg_plan_histogram_rebucket(tg_engine* h, tg_plan* p, const char* table_name, int32_t agg_index, uint64_t* counts, int32_t n_buckets) {
    return guard([&] {
        if (!h || !p || !table_name) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        Table* t = nullptr;
        {
            std::lock_guard<std::mutex> g(h->e.mu);
            auto it = h->e.tables.find(table_name);
            if (it != h->e.tables.end()) t = it->second.get();
        }
        if (!t) throw Error(TG_ERR_TABLE_NOT_FOUND, std::string("Error during planning: table 'datafusion.public.") + table_name + "' not found");
        hist_rebucket(h->e, t, p->p, agg_index, counts, n_buckets);
    });
}
tg_status tg_plan_histogram_install(tg_plan* p, int32_t agg_index, const uint64_t* counts, int32_t n_buckets) {
    return guard([&] {
        if (!p) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        p->p.histogram_install(agg_index, counts, n_buckets);
    });
}

int32_t tg_format_f64_json(double v, char* buf, int32_t cap) {
    const std::string s = json_f64(v);
    if (buf && cap > 0) {
        const size_t n = std::min<size_t>(s.size(), (size_t)cap - 1);
        memcpy(buf, s.data(), n);
        buf[n] = 0;
    }
    return (int32_t)s.size();
}

int32_t tg_plan_analyzer_state_json(const tg_plan* p, int32_t slot, char* buf, int32_t cap) {
    int32_t need = -1;
    tg_status st = guard([&] {
        if (!p) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        const std::string s = analyzer_state_json(p->p, slot);
        need = (int32_t)s.size();
        if (buf && cap > 0) {
            const size_t n = std::min<size_t>(s.size(), (size_t)cap - 1);
            memcpy(buf, s.data(), n);
            buf[n] = 0;
        }
    });
    return st == TG_OK ? need : -(int32_t)st;
}

tg_status tg_plan_redirect_aggregate(tg_plan* p, int32_t i, int32_t which, const char* table_name) {
    return guard([&] {
        if (!p || i < 0 || i >= (int32_t)p->p.aggs.size()) throw Error(TG_ERR_INVALID_ARG, "aggregate index out of range");
        Agg& a = p->p.aggs[i];
        if (which < 0 || which > 1 || (which == 1 && a.kind != A_FK) || (a.kind != A_FK && a.kind != A_DISTINCT && a.kind != A_SPEARMAN))
            throw Error(TG_ERR_INVALID_ARG, "only DISTINCT / SPEARMAN (which = 0) and FK (which = 0 child, 1 parent) aggregates can be redirected");
        if (table_name && *table_name) validate_identifier(table_name);
        a.redirect[which] = table_name ? table_name : "";
    });
}

tg_status tg_plan_result(const tg_plan* p, int32_t slot, tg_result* out) {
    return guard([&] {
        if (!p || !out) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        if (slot < 0 || slot >= (int32_t)p->p.slots.size()) throw Error(TG_ERR_INVALID_ARG, "slot out of range");
        if (!p->p.executed) throw Error(TG_ERR_INVALID_ARG, "plan has not been executed");
        const Slot& s = p->p.slots[slot];
        out->status = s.status;
        out->has_metric = s.has_metric;
        out->metric = s.metric;
        out->message = s.has_message ? s.message.c_str() : nullptr;
        out->name = s.name.c_str();
        out->error_code = 0;
        for (int a : s.aggs)
            if (p->p.aggs[a].err != TG_OK && s.kind != SL_SQL) out->error_code = p->p.aggs[a].err;
        out->reserved = 0;
    });
}

tg_status tg_plan_analyzer_result(const tg_plan* p, int32_t slot, tg_analyzer_result* out) {
    return guard([&] {
        if (!p || !out) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        if (slot < 0 || slot >= (int32_t)p->p.slots.size()) throw Error(TG_ERR_INVALID_ARG, "slot out of range");
        if (!p->p.executed) throw Error(TG_ERR_INVALID_ARG, "plan has not been executed");
        const Slot& s = p->p.slots[slot];
        if (s.kind != SL_ANALYZER && s.kind != SL_KLL && s.kind != SL_GROUPED && s.kind != SL_HISTOGRAM && s.kind != SL_VALUE_HIST)
            throw Error(TG_ERR_INVALID_ARG, "slot is not an analyzer");
        *out = s.ares;
        out->metric_key = s.metric_key.c_str();
        out->message = s.has_message ? s.message.c_str() : nullptr;
    });
}

int32_t tg_plan_map_size(const tg_plan* p, int32_t slot) {
    if (!p || slot < 0 || slot >= (int32_t)p->p.slots.size()) return -1;
    return (int32_t)p->p.slots[slot].map.size();
}
tg_status tg_plan_map_entry(const tg_plan* p, int32_t slot, int32_t i, const char** key, double* value) {
    return guard([&] {
        if (!p || slot < 0 || slot >= (int32_t)p->p.slots.size()) throw Error(TG_ERR_INVALID_ARG, "slot out of range");
        const Slot& s = p->p.slots[slot];
        if (i < 0 || i >= (int32_t)s.map.size()) throw Error(TG_ERR_INVALID_ARG, "map index out of range");
        if (key) *key = s.map[i].first.c_str();
        if (value) *value = s.map[i].second;
    });
}

tg_status tg_plan_exec_stats(const tg_plan* p, tg_exec_stats* out) {
    return guard([&] {
        if (!p || !out) throw Error(TG_ERR_INVALID_ARG, "NULL argument");
        *out = p->p.stats;
    });
}

// ------------------------------------------------------------------ host helpers ----
int32_t tg_assertion_evaluate(tg_assertion a, double value) { return assertion_evaluate(a, value) ? 1 : 0; }
static int32_t copy_out(const std::string& s, char* buf, int32_t cap) {
    if (buf && cap > 0) {
        size_t n = std::min((size_t)cap - 1, s.size());
        memcpy(buf, s.data(), n);
        buf[n] = 0;
    }
    return (int32_t)s.size();
}
int32_t tg_assertion_description(tg_assertion a, char* buf, int32_t cap) {
    return copy_out(assertion_description(a), buf, cap);
}
int32_t tg_logical_evaluate(int32_t op, int32_t n, const uint8_t* results, int32_t n_results) {
    std::vector<bool> v;
    for (int32_t i = 0; i < n_results; ++i) v.push_back(results[i] != 0);
    return logical_evaluate(op, n, v) ? 1 : 0;
}
tg_status tg_validate_identifier(const char* id) {
    return guard([&] { validate_identifier(id ? id : ""); });
}
tg_status tg_validate_regex_pattern(const char* pattern) {
    return guard([&] {
        std::string p = pattern ? pattern : "";
        validate_regex_pattern_text(p);
        (void)compile_regex(p, false);
    });
}
tg_status tg_validate_sql_expression(const char* e) {
    return guard([&] { validate_sql_expression(e ? e : ""); });
}
const char* tg_format_pattern(int32_t kind, const char* arg, int32_t flag) {
    static thread_local std::string s;
    try {
        s = format_pattern(kind, arg, flag);
    } catch (Error& e) {
        fail(e.code, e.msg);
        return nullptr;
    }
    return s.c_str();
}
int32_t tg_regex_host_match(const char* pattern, int32_t icase, const uint8_t* s, int64_t len, int32_t* out) {
    return (int32_t)guard([&] {
        Dfa d = compile_regex(pattern ? pattern : "", icase != 0);
        if (out) *out = d.match(s, len) ? 1 : 0;
    });
}
int32_t tg_regex_dfa_size(const char* pattern, int32_t icase, uint32_t* n_states, uint32_t* n_classes) {
    return (int32_t)guard([&] {
        Dfa d = compile_regex(pattern ? pattern : "", icase != 0);
        if (n_states) *n_states = d.n_states;
        if (n_classes) *n_classes = d.n_classes;
    });
}
int32_t tg_format_f64(double v, char* buf, int32_t cap) { return copy_out(fmt_f64(v), buf, cap); }

}  // extern "C"
