/*
 * termgpu.h — C ABI of the B200-native evaluator for term-guard's constraint / analyzer hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b). Every entry point below replaces the body of one
 * reference trait method that today lowers to `ctx.sql(..).collect()`; the reference file:line each
 * one stands in for is cited beside it (paths relative to the reference checkout, term-guard/src/...).
 * A Rust shim (`term-guard-gpu-sys`, see INTEGRATION.md) binds these 1:1 and implements
 * `Constraint::evaluate` (core/constraint.rs:186-225) and `Analyzer::compute_state_from_data`
 * (analyzers/traits.rs:65-148) on top of them.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types cross this boundary
 *   - every function returns tg_status; the message for the last failure on the calling thread is
 *     tg_last_error(). Data-shape problems found while evaluating (missing column, type mismatch)
 *     do NOT fail the call: like the reference (core/suite.rs:231-256) they become a failed
 *     constraint whose message starts with "Error evaluating constraint:".
 *   - the engine owns device buffers; results are POD copied out; message pointers stay valid
 *     until the owning plan is destroyed or re-executed.
 *   - there is no CPU fallback: without a CUDA device tg_engine_create fails with TG_ERR_CUDA.
 */
#ifndef TERMGPU_H
#define TERMGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TG_API __attribute__((visibility("default")))

typedef struct tg_engine tg_engine;
typedef struct tg_table tg_table;
typedef struct tg_plan tg_plan;

/* mirrors TermError variants (error.rs:16-140) as codes */
typedef enum {
    TG_OK = 0,
    TG_ERR_INVALID_ARG = 1,
    TG_ERR_COLUMN_NOT_FOUND = 2,
    TG_ERR_TYPE_MISMATCH = 3,
    TG_ERR_SECURITY = 4,      /* TermError::SecurityError (security.rs) */
    TG_ERR_UNSUPPORTED = 5,   /* syntax outside the declared regex / predicate grammar */
    TG_ERR_CUDA = 6,
    TG_ERR_NCCL = 7,
    TG_ERR_INTERNAL = 8,
    TG_ERR_TABLE_NOT_FOUND = 9,
    TG_ERR_VALIDATION = 10,   /* TermError::ValidationFailed at construction (e.g. threshold range) */
    TG_ERR_CONFIGURATION = 11 /* TermError::Configuration */
} tg_status;

typedef enum {
    TG_INT64 = 1,
    TG_FLOAT64 = 2,
    TG_UTF8 = 3,   /* Arrow Utf8: int32 offsets + value bytes */
    TG_INT32 = 4,
    TG_FLOAT32 = 5,
    TG_BOOL = 6,   /* Arrow Boolean: bit-packed values */
    TG_FP128 = 7,  /* internal: 24-byte records {h1, h2, null flag} of a hash-shuffled Utf8 / composite key
                      (tg_table_partition_fingerprints); only COUNT(DISTINCT ..)-type aggregates read it */
    TG_PQ_INT96 = 8 /* tg_table_append_parquet_chunk only: a Parquet INT96 (legacy timestamp) chunk, stored as a TG_INT64
                       column of nanoseconds since the epoch, delivered as Timestamp(Nanosecond, None); no other entry point accepts it */
} tg_dtype;

/* ConstraintStatus (core/constraint.rs:11-20) */
typedef enum { TG_SUCCESS = 0, TG_FAILURE = 1, TG_SKIPPED = 2 } tg_constraint_status;

/* Assertion (constraints/assertion.rs:13-31) */
typedef enum {
    TG_ASSERT_EQUALS = 0,
    TG_ASSERT_NOT_EQUALS = 1,
    TG_ASSERT_GREATER_THAN = 2,
    TG_ASSERT_GREATER_THAN_OR_EQUAL = 3,
    TG_ASSERT_LESS_THAN = 4,
    TG_ASSERT_LESS_THAN_OR_EQUAL = 5,
    TG_ASSERT_BETWEEN = 6,
    TG_ASSERT_NOT_BETWEEN = 7
} tg_assertion_kind;

typedef struct {
    int32_t kind; /* tg_assertion_kind */
    double a;     /* value, or lower bound */
    double b;     /* upper bound for (NOT_)BETWEEN */
} tg_assertion;

/* LogicalOperator (core/logical.rs:16-27) */
typedef enum { TG_OP_ALL = 0, TG_OP_ANY = 1, TG_OP_EXACTLY = 2, TG_OP_AT_LEAST = 3, TG_OP_AT_MOST = 4 } tg_logical_op;

/* StatisticType (constraints/statistics.rs:24-45) */
typedef enum {
    TG_STAT_MIN = 0,
    TG_STAT_MAX = 1,
    TG_STAT_MEAN = 2,
    TG_STAT_SUM = 3,
    TG_STAT_STDDEV = 4,
    TG_STAT_VARIANCE = 5,
    TG_STAT_MEDIAN = 6,     /* APPROX_PERCENTILE_CONT in the reference; KLL-backed here (SURVEY §8f.3) */
    TG_STAT_PERCENTILE = 7
} tg_stat_kind;

/* FormatType (constraints/format.rs:189-215) */
typedef enum {
    TG_FMT_REGEX = 0,
    TG_FMT_EMAIL = 1,
    TG_FMT_URL = 2,          /* flag = allow_localhost */
    TG_FMT_CREDIT_CARD = 3,  /* flag = detect_only */
    TG_FMT_PHONE = 4,        /* arg = country or NULL */
    TG_FMT_POSTAL_CODE = 5,  /* arg = country */
    TG_FMT_UUID = 6,
    TG_FMT_IPV4 = 7,
    TG_FMT_IPV6 = 8,
    TG_FMT_JSON = 9,
    TG_FMT_ISO8601 = 10,
    TG_FMT_SSN = 11
} tg_format_kind;

/* FormatOptions (constraints/format.rs:367-384) */
typedef struct {
    int32_t case_sensitive;    /* default 1 */
    int32_t trim_before_check; /* default 0 */
    int32_t null_is_valid;     /* default 1 */
} tg_format_options;

/* UniquenessType / NullHandling (constraints/uniqueness.rs:40-170) */
typedef enum {
    TG_UNIQ_FULL = 0,
    TG_UNIQ_DISTINCTNESS = 1,
    TG_UNIQ_UNIQUE_VALUE_RATIO = 2,
    TG_UNIQ_PRIMARY_KEY = 3,
    TG_UNIQ_WITH_NULLS = 4,
    TG_UNIQ_COMPOSITE = 5
} tg_uniqueness_kind;
typedef enum { TG_NULLS_EXCLUDE = 0, TG_NULLS_INCLUDE = 1, TG_NULLS_DISTINCT = 2 } tg_null_handling;

/* CorrelationValidation / CorrelationType (constraints/correlation.rs:20-90) */
typedef enum {
    TG_CORR_PEARSON = 0,
    TG_CORR_COVARIANCE = 1,
    TG_CORR_INDEPENDENCE = 2, /* ABS(CORR) <= max_correlation; assertion.a = max */
    TG_CORR_SPEARMAN = 3,     /* constraint form is Skipped in the reference (correlation.rs:340-345) */
    TG_CORR_KENDALL = 4,
    TG_CORR_MUTUAL_INFORMATION = 5,
    TG_CORR_RANGE = 6         /* Pearson with Between(a,b), name "correlation_range" */
} tg_correlation_kind;

/* analyzers (analyzers/basic/ *.rs and analyzers/advanced/{standard_deviation,correlation,kll_sketch}.rs) */
typedef enum {
    TG_AN_SIZE = 0,
    TG_AN_COMPLETENESS = 1,
    TG_AN_DISTINCTNESS = 2,
    TG_AN_MEAN = 3,
    TG_AN_MIN = 4,
    TG_AN_MAX = 5,
    TG_AN_SUM = 6,
    TG_AN_STDDEV = 7,
    TG_AN_CORR_PEARSON = 8,
    TG_AN_CORR_SPEARMAN = 9,
    TG_AN_COVARIANCE = 10,
    TG_AN_KLL = 11,
    TG_AN_GROUPED_COMPLETENESS = 12,
    TG_AN_COMPLIANCE = 13,
    TG_AN_APPROX_COUNT_DISTINCT = 14 /* analyzers/advanced/approx_count_distinct.rs; answered EXACTLY */
} tg_analyzer_kind;

/* ConstraintResult (core/constraint.rs:40-48) */
typedef struct {
    int32_t status;      /* tg_constraint_status */
    int32_t has_metric;  /* Option<f64> discriminant */
    double metric;
    const char* message; /* NULL when Option<String> is None */
    const char* name;    /* Constraint::name() */
    int32_t error_code;  /* != 0: the reference's evaluate() returns Err(..) here; status is FAILURE and
                            message is "Error evaluating constraint: ..." as core/suite.rs:231-256 reports it */
    int32_t reserved;
} tg_result;

/*
 * Analyzer state + metric. `u`/`f` hold the reference *State struct fields in declaration order:
 *   SIZE                u[0]=count                                   (analyzers/basic/size.rs)
 *   COMPLETENESS        u[0]=total_count u[1]=non_null_count         (basic/completeness.rs:58-62)
 *   DISTINCTNESS        u[0]=total_count(non-null) u[1]=distinct     (basic/distinctness.rs:57-61)
 *   MEAN                f[0]=sum u[0]=count                          (basic/mean.rs:58-62)
 *   MIN/MAX             f[0]=min f[1]=max u[0]=has_min u[1]=has_max  (basic/min_max.rs)
 *   SUM                 f[0]=sum u[0]=has_values                     (basic/sum.rs)
 *   STDDEV              u[0]=count f[0]=sum f[1]=sum_squared f[2]=mean   (advanced/standard_deviation.rs:60-75)
 *   CORR / COVARIANCE   u[0]=n f[0..5]=sum_x,sum_y,sum_x2,sum_y2,sum_xy  (advanced/correlation.rs:42-62)
 *   KLL                 u[0]=count f[0]=min f[1]=max; quantiles via tg_plan_map_*
 *   COMPLIANCE          u[0]=satisfied u[1]=total
 *   APPROX_COUNT_DISTINCT u[0]=approx_distinct_count u[1]=total_count   (advanced/approx_count_distinct.rs:59-64)
 * metric_kind: 0 Double, 1 Long, 2 Map (entries via tg_plan_map_*), 3 none (AnalyzerError::NoData)
 */
typedef struct {
    uint64_t u[4];
    double f[8];
    int32_t metric_kind;
    int32_t error;        /* 0 ok; 1 NoData; 2 InvalidData (message set) */
    double metric_double;
    int64_t metric_long;
    const char* metric_key; /* Analyzer::metric_key() */
    const char* message;
} tg_analyzer_result;

/* ---------------------------------------------------------------- engine ---- */

/* Opens CUDA device `device`, creates streams + pinned staging ring. Replaces SessionContext as the
 * owner of registered data (core/context.rs:16-39). */
TG_API tg_status tg_engine_create(int device, tg_engine** out);
TG_API void tg_engine_destroy(tg_engine* eng);
TG_API const char* tg_last_error(void);
TG_API const char* tg_version(void);
/* number of kernels this library has launched on this engine since creation (bench `gpu_launches`) */
TG_API uint64_t tg_engine_launch_count(const tg_engine* eng);
/* Waits until every host->device copy queued by tg_table_append_* has completed: after it returns the caller may free or
 * reuse the pinned host buffers it appended from. */
TG_API tg_status tg_engine_sync_copies(tg_engine* eng);
/* raw CUDA stream (cudaStream_t) the engine launches scan kernels on; for event timing by the harness */
TG_API void* tg_engine_stream(tg_engine* eng);

/* ---------------------------------------------------------------- tables ---- */

/* SessionContext::register_table(name, MemTable) — creates an empty table; columns are appended
 * batch by batch like RecordBatches of a MemTable partition. */
TG_API tg_status tg_table_create(tg_engine* eng, const char* name, tg_table** out);
TG_API tg_status tg_table_drop(tg_engine* eng, const char* name);
TG_API tg_status tg_table_lookup(tg_engine* eng, const char* name, tg_table** out);
TG_API int64_t tg_table_num_rows(const tg_table* t);
/* schema lookup (SessionContext::table(..).schema().field_with_name(..).data_type()) -> tg_dtype */
TG_API tg_status tg_table_column_dtype(const tg_table* t, const char* column, int32_t* dtype);
/* Device addresses of a column's Arrow buffers (engine-owned, valid until the table is dropped or appended to; all
 * pending host->device copies of the engine are complete on return). validity / offsets are NULL when the column has
 * none. Used by the multi-GPU host code to move a column between ranks (SURVEY §8e, K6: Spearman's global ranks). */
typedef struct tg_column_buffers {
    int32_t dtype;
    int64_t n_rows;
    const void* values;
    const void* offsets;
    const void* validity;
    int64_t n_value_bytes;
    int64_t null_count;
} tg_column_buffers;
TG_API tg_status tg_table_column_buffers(tg_engine* eng, const char* table, const char* column, tg_column_buffers* out);

/*
 * Parquet column chunk -> HBM (SURVEY §8f.4): replaces the decode of the reference's ParquetSource
 * (sources/parquet.rs:150-230, DataFusion ParquetExec -> Arrow RecordBatch) and the host->device copy for one
 * column. `chunk` = the column chunk's bytes exactly as they are in the file (from the first page header,
 * total_compressed_size bytes), `num_values` / `codec` / the physical type (as tg_dtype) / the leaf's max definition
 * level from the file metadata. The host walks the page headers and expands the definition levels into the validity
 * bitmap while the value bytes travel; compressed pages are inflated on the host (Snappy by the library's own decoder, GZIP /
 * BROTLI / ZSTD / LZ4_RAW by the host's codec libraries, bound at run time); the device scatters the densely stored
 * non-NULL values to their rows, looking dictionary-encoded ones up through the page's index stream (RLE / bit-packed
 * hybrid, only its run headers are walked on the host) and the chunk's dictionary.
 * BYTE_ARRAY strings (dtype TG_UTF8) become int32 offsets + concatenated bytes: the device locates every row's bytes
 * (dictionary entry or PLAIN value), scans the lengths and copies; the host walks the PLAIN pages' length prefixes.
 * BOOLEAN (dtype TG_BOOL) becomes the bit-packed Arrow Boolean values; its PLAIN and RLE values are decoded on the device.
 * INT96 (dtype TG_PQ_INT96, the legacy Impala / Hive / Spark timestamp: int64 nanoseconds of the day, int32 Julian day)
 * becomes an Int64 column of nanoseconds since the epoch (wrapping outside 1677 .. 2262), declared Timestamp(Nanosecond,
 * None) by this call; appending it to a column of another delivered type is TG_ERR_TYPE_MISMATCH.
 * Supported: INT64 / DOUBLE / INT32 / FLOAT / INT96 / BOOLEAN / BYTE_ARRAY (Utf8), codec UNCOMPRESSED (0) / SNAPPY (1) / GZIP (2) / BROTLI (4) / ZSTD (6) /
 * LZ4_RAW (7) (parquet.thrift CompressionCodec numbers; LZO and the deprecated hadoop-framed LZ4 are refused), data
 * pages V1 / V2, PLAIN / PLAIN_DICTIONARY / RLE_DICTIONARY values (on the device; BOOLEAN: PLAIN / RLE) and DELTA_BINARY_PACKED /
 * DELTA_LENGTH_BYTE_ARRAY / DELTA_BYTE_ARRAY / BYTE_STREAM_SPLIT values of INT64 / DOUBLE / INT32 / FLOAT / BYTE_ARRAY (serial streams:
 * rewritten to PLAIN on the host), RLE levels, flat columns; anything else -> TG_ERR_UNSUPPORTED (there is no host decode path).
 * Appends num_values rows; `chunk`
 * must stay readable until the next tg_plan_execute* / tg_table_column_buffers on this engine when it is pinned memory.
 * A failed call leaves the table as it was (no column created, no type declared).
 */
TG_API tg_status tg_table_append_parquet_chunk(tg_table* t, const char* name, int32_t dtype, int32_t max_definition_level,
                                               int32_t codec, const void* chunk, int64_t n_bytes, int64_t num_values);
/* Declares the Arrow type (C Data Interface format string) that a stored Int32 / Int64 column stands for when its values
 * arrived already in the stored representation — Parquet chunks annotated DATE ("tdD"), TIME ("ttm" / "ttu" / "ttn"),
 * TIMESTAMP ("tsm:" / "tsu:" / "tsn:"), INT(8|16, signed) ("c" / "s"), INT(8|16, unsigned) ("C" / "S"): the physical values are
 * the Arrow values. The column then follows the typing rules of tg_table_append_arrow for that type (temporal columns:
 * comparisons / completeness / uniqueness / grouping; MIN / MAX / SUM result types as DataFusion's, sources/parquet.rs:150-230
 * yields these logical Arrow types). UInt32 / UInt64 need converted values and are refused here. */
TG_API tg_status tg_table_set_column_arrow_type(tg_table* t, const char* column, const char* arrow_format);
/* Host-only page walk of a column chunk (Thrift compact PageHeaders, parquet.thrift): fills up to `cap` entries and
 * returns the number of pages, or -(tg_status). page_type: 0 DATA_PAGE, 1 INDEX_PAGE, 2 DICTIONARY_PAGE, 3 DATA_PAGE_V2 */
typedef struct tg_parquet_page {
    int32_t page_type, version;
    int32_t encoding, definition_level_encoding;
    int32_t num_values, num_nulls;
    int32_t uncompressed_bytes, body_bytes;
    int32_t definition_levels_bytes, repetition_levels_bytes;
    int32_t is_compressed, reserved;
    int64_t header_offset, body_offset;
} tg_parquet_page;
TG_API int32_t tg_parquet_inspect_chunk(const void* chunk, int64_t n_bytes, tg_parquet_page* pages, int32_t cap);
/* Host-only: expands the definition levels of a flat optional column chunk into `out_bits` ((num_values + 7) / 8 bytes,
 * LSB first, chunk-relative; may be NULL) and returns the non-NULL count, or -(tg_status). The bitmap the device path uses. */
TG_API int64_t tg_parquet_chunk_validity(const void* chunk, int64_t n_bytes, int64_t num_values, uint8_t* out_bits);
/* Host-only: the Snappy raw-format decoder the chunk path applies to compressed pages (parquet-format Compression.md);
 * returns the uncompressed size, or -(tg_status) for a corrupt stream / a stream larger than `cap`. */
TG_API int64_t tg_parquet_snappy_decompress(const void* src, int64_t n_bytes, void* dst, int64_t cap);
/* Host-only: the value section of one data page (n_values non-NULL values) encoded DELTA_BINARY_PACKED (5), DELTA_LENGTH_BYTE_ARRAY
 * (6), DELTA_BYTE_ARRAY (7) or BYTE_STREAM_SPLIT (9) (parquet.thrift Encoding numbers) rewritten into the PLAIN layout
 * (elem_width 4 / 8: little-endian values; 0: BYTE_ARRAY as 4-byte length + bytes) — what the chunk path does on the host for
 * such pages before the common PLAIN path stages them. Returns the PLAIN size, or -(tg_status). */
TG_API int64_t tg_parquet_decode_to_plain(int32_t encoding, int32_t elem_width, const void* src, int64_t n_bytes, int64_t n_values, void* dst,
                                          int64_t cap);
/* Host-only: one compressed page body of codec `codec` (parquet.thrift numbers, see above) -> dst; returns the uncompressed
 * size, or -(tg_status): TG_ERR_UNSUPPORTED for a codec without a decoder (or whose library this host lacks),
 * TG_ERR_INVALID_ARG for a corrupt stream / one larger than `cap`. What the chunk path applies to every compressed page. */
TG_API int64_t tg_parquet_page_decompress(int32_t codec, const void* src, int64_t n_bytes, void* dst, int64_t cap);

/*
 * Append `n_rows` rows to column `name` from HOST Arrow buffers (values / int32 offsets / validity
 * bitmap, LSB bit order, `bit_offset` = Arrow array offset). The call stages them through pinned
 * memory into HBM (async copies on the engine's copy stream) and returns after the copy is queued and
 * the caller's buffers are no longer needed. validity may be NULL (no nulls). For TG_UTF8 `values`
 * is the byte buffer and `offsets` has n_rows+1 entries. First call for a name defines its dtype. A failed call leaves the
 * table as it was.
 */
TG_API tg_status tg_table_append_host(tg_table* t, const char* name, int32_t dtype, int64_t n_rows,
                                      const void* values, const int32_t* offsets,
                                      const uint8_t* validity, int64_t bit_offset);

/*
 * Adopt DEVICE-resident Arrow buffers without copying (HBM-resident path). Pointers must be 16-byte
 * aligned and readable up to the next multiple of 16 bytes. The engine does not take ownership.
 * `n_value_bytes` is the Utf8 byte-buffer length (ignored otherwise).
 */
TG_API tg_status tg_table_adopt_device(tg_table* t, const char* name, int32_t dtype, int64_t n_rows,
                                       const void* d_values, const int32_t* d_offsets,
                                       const uint8_t* d_validity, int64_t n_value_bytes);

/*
 * Multi-GPU hash shuffle, step 1 (SURVEY.md §8e; stands where DataFusion's RepartitionExec(Hash) stands under
 * COUNT(DISTINCT ..) / the foreign-key LEFT JOIN, constraints/uniqueness.rs:549-718, foreign_key.rs:165-172).
 * Groups the valid (non-NULL) keys of an Int64 / Float64 column by destination part = f(hash(key)), so that equal
 * keys of every rank meet on one rank after an all-to-all. *d_keys receives a DEVICE pointer to the keys (raw
 * 64-bit values, part 0 first; valid until the next call of this function on the engine), counts[n_parts] the
 * keys per part, *n_null_rows the NULL rows (the host layer sends them to part 0 as a count). The all-to-all
 * itself is the host layer's (NCCL); the receiving rank adopts the keys as a table (tg_table_adopt_device) and
 * runs the ordinary plan on it — the partial states of hash-disjoint shards merge by addition.
 */
TG_API tg_status tg_table_partition_keys(tg_engine* eng, const char* table, const char* column, int32_t n_parts,
                                         void** d_keys, int64_t* counts, int64_t* n_null_rows);

/* Same for Utf8 and composite keys: every row's key tuple is reduced to its 128-bit fingerprint (the identity the
 * single-GPU path uses too) plus a "has a NULL component" flag, and the 24-byte records {h1, h2, flag} are grouped
 * by destination part. The receiving rank adopts them as ONE column named "tg_fp" of dtype TG_FP128 and redirects
 * the DISTINCT aggregate to that table. (Foreign keys over Utf8 columns stay single-GPU: their violation examples
 * need the strings.) */
TG_API tg_status tg_table_partition_fingerprints(tg_engine* eng, const char* table, const char* const* columns,
                                                 int32_t n_columns, int32_t n_parts, void** d_records, int64_t* counts);

/*
 * The shuffle as ONE call, NCCL inside the library (libnccl.so.2 is bound at run time, so single-GPU hosts never load it).
 * One communicator per engine: rank 0 calls tg_comm_unique_id, the host carries the 128 bytes to every rank (any
 * transport), every rank calls tg_comm_init (collective, like ncclCommInitRank). tg_table_shuffle_column then does, for
 * one Int64 / Float64 key column: partition the valid keys by destination rank on the device, all-gather the counts,
 * ncclSend / ncclRecv every part (one group) straight into the value buffer of a NEW engine-owned table `shard_table`
 * (same column name; the NULL rows of every rank become trailing NULL rows of rank 0's shard) — what
 * tg_table_partition_keys + a host-side all-to-all + tg_table_adopt_device do in three steps. The aggregate is then
 * redirected to the shard (tg_plan_redirect_aggregate) and the shard dropped with tg_table_drop after the step. On one
 * node the transfer is not even a separate step: the ranks' receive buffers are mapped into every peer through CUDA IPC
 * and the partition's scatter kernel writes each part straight into its destination over NVLink ("push shuffle").
 * tg_table_shuffle_fingerprints: the same for Utf8 / composite keys (24-byte records, column "tg_fp", dtype TG_FP128).
 * tg_comm_bytes_sent: bytes this rank has sent to other ranks through these calls (bench bookkeeping).
 */
TG_API tg_status tg_comm_unique_id(void* id128);
TG_API tg_status tg_comm_init(tg_engine* eng, const void* id128, int32_t world, int32_t rank);
TG_API tg_status tg_comm_destroy(tg_engine* eng);
TG_API uint64_t tg_comm_bytes_sent(const tg_engine* eng);
/* partition: 0 = by hash (the only choice for a foreign key: both sides must use the same function); 1 = by value range when
 * the Int64 keys are globally dense (decided from the all-gathered min / max / count, abandoned when the slices come
 * out unbalanced), by hash otherwise — a rank's slice of a dense key space de-duplicates on the L2-resident bitmap path. */
TG_API tg_status tg_table_shuffle_column(tg_engine* eng, const char* table, const char* column, const char* shard_table,
                                         int32_t partition, int64_t* n_rows);
TG_API tg_status tg_table_shuffle_fingerprints(tg_engine* eng, const char* table, const char* const* columns, int32_t n_columns,
                                               const char* shard_table, int64_t* n_rows);

/* Arrow C Data Interface ingestion: `schema`/`array` are struct ArrowSchema* / struct ArrowArray* of a
 * struct-typed array (a RecordBatch). The engine copies; the caller keeps ownership and releases.
 * String encodings: Utf8 ("u"), LargeUtf8 ("U"), Utf8View ("vu") and dictionaries with any integer index type ("c" .. "L")
 * over Utf8 / LargeUtf8 values are all stored as one Utf8 column of the logical values (batches of a column may mix them,
 * each with its own dictionary; array offsets on the column and on the dictionary are honoured). Views and dictionaries
 * cross PCIe encoded and are decoded on the device. A row is NULL when its validity bit is clear or its index names a
 * NULL dictionary value; indices and views under NULL rows are never read. Errors: TG_ERR_INVALID_ARG for a valid row whose
 * index lies outside the dictionary (any valid row of an empty one) or whose view lies outside its data buffer;
 * TG_ERR_UNSUPPORTED for a string of 16 MiB or more, for BinaryView ("vz") and for dictionaries of any other value type
 * (Binary, Utf8View, numeric, temporal, Boolean). A failed call leaves the table as it was: no column holds any of the
 * batch's rows. */
TG_API tg_status tg_table_append_arrow(tg_table* t, const void* arrow_schema, const void* arrow_array);

/* Arrow C Device Data Interface ingestion: `arrow_device_array` is a struct ArrowDeviceArray* (128 bytes: the ArrowArray,
 * int64 device_id, int32 device_type at byte 88, void* sync_event at byte 96, reserved) of a struct-typed array (a
 * RecordBatch); `arrow_schema` as for tg_table_append_arrow. The caller keeps ownership; the engine never calls release.
 * By device_type:
 *   CPU (1): tg_table_append_arrow.
 *   CUDA_HOST (3): tg_table_append_arrow, after cudaEventSynchronize(*(cudaEvent_t*)sync_event) when an event is given.
 *   CUDA (2), CUDA_MANAGED (13): converted in HBM by copies and kernels on the engine's device. device_id must be the
 *     engine's device (TG_ERR_INVALID_ARG otherwise); a given sync_event (a cudaEvent_t*) is waited for on the device
 *     before any work. Before any copy or kernel, every buffer is checked with cudaPointerGetAttributes: device or managed
 *     memory of the engine's device only (a host pointer labelled CUDA, or another GPU's memory: TG_ERR_INVALID_ARG). The
 *     Utf8View variadic-sizes buffer may be host or device memory. Index, offset and value buffers read by a kernel must be
 *     aligned to their element size (TG_ERR_INVALID_ARG otherwise).
 *   Any other device type: TG_ERR_UNSUPPORTED.
 * Types, results and errors are those of tg_table_append_arrow: the call leaves exactly the state a host append of the same
 * batch leaves, and a failed call leaves the table as it was. The call returns only after every copy and kernel that reads
 * the producer's buffers has finished: the producer may free or reuse them as soon as it returns. */
TG_API tg_status tg_table_append_arrow_device(tg_table* t, const void* arrow_schema, const void* arrow_device_array);

/*
 * CSV -> HBM: replaces the reference's CsvSource::register -> DataFusion CSV scan (arrow-csv) -> Arrow batches -> H2D for
 * the GPU path. `bytes` = the file's bytes, or any run of whole records (the caller maps the file; the engine does no I/O).
 * Columns are given by the caller's schema, in file order: name + Arrow C Data Interface format string — "l" Int64, "i"
 * Int32, "g" Float64, "b" Boolean, "u" Utf8, "tdD" Date32, "tss:" / "tsm:" / "tsu:" / "tsn:" naive Timestamp (temporal columns
 * are declared as tg_table_set_column_arrow_type declares them); any other format is TG_ERR_UNSUPPORTED, naming the type.
 * Format: records end at LF, CRLF or a lone CR, blank lines are skipped, the last record needs no terminator; `delimiter` is
 * one byte, the quote is '"' (RFC 4180: it opens quoting at a field's start only, "" inside quotes is a quote, bytes after
 * the closing quote are kept); `has_header` skips the first record without checking its names. An empty field, quoted or
 * not, is NULL for every type. Values: Int64 / Int32 [+-]?[0-9]+ in range; Float64 [+-]?(d+[.d*] | .d+)([eE][+-]?d+)? and
 * nan / inf / infinity (case-insensitive, signed), correctly rounded; Boolean true / false (case-insensitive); Date32
 * YYYY-MM-DD; Timestamp YYYY-MM-DD[T| ]HH:MM:SS[.f{1,9}] (fraction digits past the unit dropped); Utf8 valid UTF-8. No
 * whitespace is trimmed. A wrong field count, an unterminated quote, a value outside its grammar or range and invalid UTF-8
 * are TG_ERR_INVALID_ARG, the message naming the line the record starts on and the column. A failed call leaves every
 * column of the table as it was; appending to a column of another type is TG_ERR_TYPE_MISMATCH. *rows_out (may be NULL):
 * the rows appended. The bytes are staged in chunks of TG_CSV_CHUNK_BYTES (default 256 MiB); a longer record grows its chunk.
 */
TG_API tg_status tg_table_append_csv(tg_table* t, const char* const* columns, const char* const* arrow_formats, int32_t n_columns,
                                     const void* bytes, int64_t n_bytes, int32_t delimiter, int32_t has_header, int64_t* rows_out);

/*
 * A CSV dialect, as arrow-csv's Format (DataFusion's CsvReadOptions: delimiter, quote, escape, comment, terminator,
 * null_regex) reads it through csv-core. Each byte field is 0..255 or -1: delimiter -1 = ','; quote -1 = '"'; escape and
 * comment -1 = none; terminator -1 = LF, CRLF or a lone CR. The delimiter, quote, escape, comment and terminator bytes must
 * be pairwise distinct (the default terminator counts as both CR and LF); a clash is TG_ERR_INVALID_ARG naming both.
 *  - quote: opens quoting at a field's start only; inside quotes a doubled quote is one quote; bytes after the closing quote
 *    are kept.
 *  - escape: only inside quotes, the escape byte and the byte after it stand for that byte (whatever it is: a quote, the
 *    escape byte, a terminator). Outside quotes it is an ordinary byte.
 *  - comment: a record whose first byte is the comment byte is skipped up to and including its terminator. The byte counts
 *    only at a record's start; comment lines before the header are skipped, the header is the first other record.
 *  - terminator: when given, only that byte ends a record and CR and LF are ordinary bytes (a CRLF file read with LF keeps
 *    the CR in its last field). Blank records are skipped with every terminator.
 *  - null_regex (NULL = none): a field is NULL when the regex finds a match in its unescaped value (unanchored search with
 *    the Rust regex crate's semantics, as arrow-csv's NullRegex::is_null). With a regex, an empty field is NULL only when
 *    the regex matches ""; otherwise it is "" in a Utf8 column and a value error in any other. Without one, an empty field
 *    is NULL. An invalid pattern is TG_ERR_INVALID_ARG; a construct the DFA compiler does not support TG_ERR_UNSUPPORTED.
 * Error messages name the line a record starts on, where a line is what the terminator ends (comment and blank lines count).
 */
typedef struct {
    int32_t delimiter, quote, escape, comment, terminator; /* -1 = none / default */
    int32_t has_header;
    const char* null_regex; /* NULL = none */
} tg_csv_format;

/* tg_table_append_csv with a CSV dialect; tg_table_append_csv is this call with {delimiter, -1, -1, -1, -1, has_header, NULL}. */
TG_API tg_status tg_table_append_csv_format(tg_table* t, const char* const* columns, const char* const* arrow_formats, int32_t n_columns,
                                            const void* bytes, int64_t n_bytes, const tg_csv_format* format, int64_t* rows_out);
/* Host-only: the tokenizer's transition table and the field rules run on the CPU (tests / diagnostics), without a schema.
 * For n_bytes of input: `values` (room for n_bytes) receives every field's unescaped bytes back to back, value_ends[i] the
 * end of field i in `values` and is_null[i] whether it is NULL (room for n_bytes + 1 fields each); record_fields[r] the
 * number of fields of record r and record_lines[r] the line it starts on (room for n_bytes + 1 records each); *n_fields and
 * *n_records (may be NULL) the counts. An unterminated quote is TG_ERR_INVALID_ARG naming its record's line. */
TG_API tg_status tg_csv_split_host(const tg_csv_format* format, const void* bytes, int64_t n_bytes, uint8_t* values, int64_t* value_ends,
                                   uint8_t* is_null, int64_t* record_fields, int64_t* record_lines, int64_t* n_fields, int64_t* n_records);
/* Host-only: the value parser the device runs, for one raw field (quoted or not) of the given format (tests / diagnostics).
 * `out` (may be NULL) receives the stored value — 8 bytes for Int64 / Float64 / Timestamp, 4 for Int32 / Date32, 1 (0 / 1)
 * for Boolean, and for Utf8 the unescaped length as an int64 — and *is_null (may be NULL) whether the field is NULL.
 * Errors as tg_table_append_csv's, without the line and column. */
TG_API tg_status tg_csv_parse_value(const char* arrow_format, const void* field, int64_t n_bytes, void* out, int32_t* is_null);

/* ------------------------------------------------------------------ plan ---- */

/* A plan is the fused form of a Check / ValidationSuite / AnalysisRunner: every add_* returns a slot
 * (>= 0) or a negative tg_status. One tg_plan_execute evaluates all slots with at most one numeric
 * pass, one pass per string column and one hash job per key set. */
TG_API tg_status tg_plan_create(tg_plan** out);
TG_API void tg_plan_destroy(tg_plan* plan);
TG_API int32_t tg_plan_num_slots(const tg_plan* plan);

/* CompletenessConstraint::new (constraints/completeness.rs:96-110), evaluate_column :137-246,
 * multi-column combine core/unified.rs:41-123 */
TG_API int32_t tg_plan_add_completeness(tg_plan* plan, const char* const* columns, int32_t n_columns,
                                        double threshold, int32_t logical_op, int32_t logical_n);
/* SizeConstraint::evaluate (constraints/size.rs:53-119) */
TG_API int32_t tg_plan_add_size(tg_plan* plan, tg_assertion assertion);
/* StatisticalConstraint::evaluate (constraints/statistics.rs:254-322) */
TG_API int32_t tg_plan_add_statistic(tg_plan* plan, const char* column, int32_t stat_kind,
                                     double percentile, tg_assertion assertion);
/* MultiStatisticalConstraint::evaluate (constraints/statistics.rs:424-504) */
TG_API int32_t tg_plan_add_multi_statistic(tg_plan* plan, const char* column, const int32_t* stat_kinds,
                                           const double* percentiles, const tg_assertion* assertions,
                                           int32_t n);
/* FormatConstraint::new / evaluate (constraints/format.rs:490-520, 740-843) */
TG_API int32_t tg_plan_add_format(tg_plan* plan, const char* column, int32_t format_kind,
                                  const char* arg, int32_t flag, double threshold,
                                  const tg_format_options* options);
/* UniquenessConstraint::new / evaluate (constraints/uniqueness.rs:262-308, 449-482) */
TG_API int32_t tg_plan_add_uniqueness(tg_plan* plan, const char* const* columns, int32_t n_columns,
                                      int32_t uniqueness_kind, double threshold, tg_assertion assertion,
                                      int32_t null_handling);
/* CorrelationConstraint::evaluate (constraints/correlation.rs:299-440) */
TG_API int32_t tg_plan_add_correlation(tg_plan* plan, const char* column1, const char* column2,
                                       int32_t correlation_kind, tg_assertion assertion);
/* CustomSqlConstraint::new / evaluate (constraints/custom_sql.rs:60-98, 195-282); hint may be NULL */
TG_API int32_t tg_plan_add_custom_sql(tg_plan* plan, const char* expression, const char* hint);
/* ForeignKeyConstraint::evaluate (constraints/foreign_key.rs:307-410); columns are "table.column" */
TG_API int32_t tg_plan_add_foreign_key(tg_plan* plan, const char* child_column, const char* parent_column,
                                       int32_t allow_nulls, int32_t max_violations_reported);

/* LengthConstraint::evaluate (constraints/length.rs:150-226); LengthAssertion (:20-60) as kind: 0 Min(a),
 * 1 Max(a), 2 Between(a, b), 3 Exactly(a), 4 NotEmpty. LENGTH counts characters, not bytes. */
typedef enum { TG_LEN_MIN = 0, TG_LEN_MAX = 1, TG_LEN_BETWEEN = 2, TG_LEN_EXACTLY = 3, TG_LEN_NOT_EMPTY = 4 } tg_length_kind;
TG_API int32_t tg_plan_add_length(tg_plan* plan, const char* column, int32_t length_kind, int64_t a, int64_t b);
/* ContainmentConstraint::evaluate (constraints/values.rs:232-296) */
TG_API int32_t tg_plan_add_containment(tg_plan* plan, const char* column, const char* const* allowed_values,
                                       int32_t n_values);
/* NonNegativeConstraint::evaluate (constraints/values.rs:357-414) */
TG_API int32_t tg_plan_add_non_negative(tg_plan* plan, const char* column);

/* ApproxCountDistinctConstraint::evaluate (constraints/approx_count_distinct.rs:49-134). APPROX_DISTINCT's
 * HyperLogLog estimate is replaced by the exact distinct count of the hash job (SURVEY §8f.3). */
TG_API int32_t tg_plan_add_approx_count_distinct(tg_plan* plan, const char* column, tg_assertion assertion);

/* DataTypeConstraint::evaluate (constraints/values.rs:104-165); DataType (:14-37) */
typedef enum { TG_DT_INTEGER = 0, TG_DT_FLOAT = 1, TG_DT_BOOLEAN = 2, TG_DT_DATE = 3, TG_DT_TIMESTAMP = 4, TG_DT_STRING = 5 } tg_value_type;
TG_API int32_t tg_plan_add_data_type(tg_plan* plan, const char* column, int32_t value_type, double threshold);

/* QuantileConstraint::evaluate (constraints/quantile.rs:282-482); QuantileValidation (:83-111) as `validation`.
 * SINGLE: one quantile + assertion (median / percentile constructors :186-203), metric = the quantile value.
 * MULTIPLE: n quantiles each with its assertion (:206-213), no metric. MONOTONIC: n quantiles, `strict` (:102-106),
 * assertions NULL. UNIMPLEMENTED: Distribution / Custom, which the reference answers Skipped (:474-479).
 * APPROX_PERCENTILE_CONT (t-digest) is answered from the column's KLL sketch (SURVEY §8f.3). */
typedef enum { TG_QUANTILE_SINGLE = 0, TG_QUANTILE_MULTIPLE = 1, TG_QUANTILE_MONOTONIC = 2, TG_QUANTILE_UNIMPLEMENTED = 3 } tg_quantile_validation;
TG_API int32_t tg_plan_add_quantile(tg_plan* plan, const char* column, int32_t validation, const double* quantiles,
                                    const tg_assertion* assertions, int32_t n, int32_t strict);

/* ColumnCountConstraint::evaluate (constraints/column_count.rs:43-85): schema width of the plan's table */
TG_API int32_t tg_plan_add_column_count(tg_plan* plan, tg_assertion assertion);
/* HistogramAnalyzer (analyzers/advanced/histogram.rs:62-358), Float64 columns like the reference. Result through
 * tg_plan_analyzer_result (u[0]=total_count f[0..3]=min,max,sum,sum_squared) and tg_plan_map_*: min, max, mean,
 * std_dev, total_count, sum, sum_squared, bucket_{i}.lower / .upper / .count. Row shards whose [min, max] differ merge through
 * the second phase below (tg_plan_histogram_pending / _rebucket / _install). */
TG_API int32_t tg_plan_add_histogram(tg_plan* plan, const char* column, int32_t num_buckets);

/* Analyzers: column2 only for the correlation kinds; expression only for COMPLIANCE. */
TG_API int32_t tg_plan_add_analyzer(tg_plan* plan, int32_t analyzer_kind, const char* column,
                                    const char* column2, const char* expression);
/* KllSketch (analyzers/advanced/kll_sketch.rs:142-400) behind the documented KllSketchAnalyzer shape
 * (docs/reference/analyzers.md:327-356): metric Map{min,max,count,quantile_{p}} */
TG_API int32_t tg_plan_add_kll(tg_plan* plan, const char* column, int32_t k, const double* quantiles,
                               int32_t n_quantiles);
/* CompletenessAnalyzer::with_grouping (analyzers/basic/grouped_completeness.rs:99-239,
 * analyzers/grouped.rs:17-59). At most 8 group columns, and at most 1048576 (2^20) groups per row shard, whatever
 * max_groups says: above either the slot's result is an error (TG_ERR_UNSUPPORTED, "grouped completeness: more than
 * 8 grouping columns" / "... more than 1048576 groups"). tg_plan_add_value_histogram has the same group limit. */
TG_API int32_t tg_plan_add_grouped_completeness(tg_plan* plan, const char* column,
                                                const char* const* group_columns, int32_t n_group_columns,
                                                int32_t max_groups, int32_t include_overall);

/* HistogramConstraint (constraints/histogram.rs:208-413): value frequencies of `column` (GROUP BY CAST(column AS VARCHAR) over
 * the non-NULL rows, ORDER BY count DESC, value). After execute: tg_plan_result gives Skipped("No data to analyze") when no
 * row is non-NULL, otherwise a provisional Success whose metric is the histogram's entropy; tg_plan_map_entry(slot, i) walks
 * the buckets in order (key = value, value = count) and tg_plan_analyzer_result's u[0..2] = {total_count, null_count,
 * distinct_count}. The HistogramAssertion is a closure: the host applies it to the buckets and, when it fails, builds the
 * reference's message (histogram.rs:371-381). Utf8, integer and Boolean columns; floating-point and temporal columns are
 * TG_ERR_UNSUPPORTED (Arrow's CAST(.. AS VARCHAR) formatting of those is not restated). At most 2^20 distinct values. */
TG_API int32_t tg_plan_add_value_histogram(tg_plan* plan, const char* column);

/*
 * Evaluate every slot against table `table_name` (the reference's task-local
 * ValidationContext::table_name, core/validation_context.rs:71-82; default "data"). Blocking.
 * Equivalent to execute_partial + finalize on one GPU.
 */
TG_API tg_status tg_plan_execute(tg_engine* eng, tg_plan* plan, const char* table_name);

/* Multi-GPU (row-partitioned) form: each rank runs execute_partial on its shard, exchanges the
 * serialised partial aggregates (a small POD blob; NCCL/gloo all-gather is done by the host layer),
 * merges every rank's blob IN RANK ORDER and finalizes — mirrors AnalyzerState::merge
 * (analyzers/traits.rs:154-179). */
TG_API tg_status tg_plan_execute_partial(tg_engine* eng, tg_plan* plan, const char* table_name);
TG_API tg_status tg_plan_partial_size(const tg_plan* plan, size_t* n_bytes);
TG_API tg_status tg_plan_partial_export(const tg_plan* plan, void* buf, size_t n_bytes);
/* host-only: build partials for a plan without a GPU from an exported blob (tests, incremental runs) */
TG_API tg_status tg_plan_partial_reset(tg_plan* plan);
TG_API tg_status tg_plan_partial_merge(tg_plan* plan, const void* buf, size_t n_bytes);
TG_API tg_status tg_plan_finalize(tg_plan* plan);
/* The de-duplicated device aggregates behind the slots, in partial-blob order: kind is one of
 * 0 ROWS, 1 VALID, 2 NUM, 3 PAIR, 4 PRED, 5 REGEX, 6 DISTINCT, 7 FK, 8 KLL, 9 GROUPED, 10 SPEARMAN, 11 LENGTH, 12 HIST; key is a
 * stable textual identity such as "num|price" (valid until the plan is destroyed). Lets a host that computed a
 * shard elsewhere (another engine, a stored IncrementalAnalysisRunner state) assemble a partial blob. */
TG_API int32_t tg_plan_num_aggregates(const tg_plan* plan);
TG_API tg_status tg_plan_aggregate_info(const tg_plan* plan, int32_t i, int32_t* kind, const char** key);

/*
 * Peer mailboxes: the per-step exchange of partial states over NVLink / NVSwitch peer memory instead of
 * H2D -> ncclAllGather -> D2H (one node, one process per GPU). Each rank creates a mailbox (a small device buffer;
 * *handle_out receives its 64-byte cudaIpcMemHandle_t), the host layer all-gathers the handles once (any transport)
 * and every rank opens them. tg_plan_exchange_and_finalize then replaces
 * export / all-gather / reset / merge-in-rank-order / finalize: one kernel stores this rank's blob into every peer's
 * mailbox and raises a flag, a second waits for all flags, one copy brings the collected blobs to the host.
 * Falls back to the NCCL path of the host layer when a blob exceeds slot_bytes (TG_ERR_INVALID_ARG).
 */
TG_API tg_status tg_engine_mailbox_create(tg_engine* eng, int32_t world, int32_t rank, size_t slot_bytes, void* handle_out);
TG_API tg_status tg_engine_mailbox_open(tg_engine* eng, const void* handles /* world x 64 bytes, rank order */);
TG_API tg_status tg_plan_exchange_and_finalize(tg_engine* eng, tg_plan* plan);
/* Same, for partial blobs of any size: when some rank's blob does not fit its mailbox slot, that rank publishes a
 * "does not fit" marker instead, EVERY rank returns *fell_back = 1 without merging anything, and the host layer
 * exchanges the blobs over NCCL (tg_plan_partial_export / _merge). */
TG_API tg_status tg_plan_exchange_ex(tg_engine* eng, tg_plan* plan, int32_t* fell_back);
/* The whole multi-GPU step of a scan-only plan (ROWS / VALID / NUM / PAIR / PRED aggregates: everything the fused
 * numeric scan answers) in one call: partial execute on this rank's shard, the aggregates' partial states assembled ON
 * THE DEVICE behind the scan (no host round trip), published into every peer's mailbox over NVLink, collected, merged in
 * rank order like AnalyzerState::merge (analyzers/traits.rs:154-179) and finalized — one stream synchronisation per
 * step. *done = 0: the plan holds other aggregates, or no mailbox is open; nothing was executed and the caller takes
 * tg_plan_execute_partial + tg_plan_exchange_ex. Every rank must call it with the same plan. */
TG_API tg_status tg_plan_execute_exchange(tg_engine* eng, tg_plan* plan, const char* table_name, int32_t* done);

/*
 * Distributed RANK() OVER (ORDER BY ..) for the Spearman analyzer across row shards (SURVEY §8e K6; the reference's
 * two window functions, analyzers/advanced/correlation.rs:334-350, see every row of the table). One rank session per
 * engine; the host layer runs a SAMPLE SORT around these stages, once per column:
 *     tg_rank_begin          the shard's pairwise-complete rows as order-preserving keys (keys = x, payload = y)
 *     tg_rank_local_sort     sort the shard by key (hand-written radix sort)
 *     tg_rank_sample         up to n evenly spaced keys of the sorted shard -> host; all ranks all-gather their samples,
 *                            sort them and take world - 1 splitters at equal steps
 *     tg_rank_split          counts[p] = keys of this shard that belong to part p = the keys in (splitter[p-1], splitter[p]]
 *     tg_rank_send_buffers / tg_rank_recv_buffers     device pointers for the all-to-all of keys and payload (NCCL);
 *                            payload_bytes is 8 in the x phase (the y key) and 4 in the y phase (rank_x)
 *     tg_rank_recv_commit    the received range becomes the session's data
 *     tg_rank_finish_x       sort the range by x; minimum rank of a key = rank_base + position of its run's head + 1 with
 *                            rank_base = number of keys on the lower ranks; the data becomes (keys = y, payload = rank_x)
 *     tg_rank_finish_y       same by y; returns the range's pair count and the sums of (rank_x - c), (rank_y - c), their
 *                            squares and their product, c = `center` = (N + 1) / 2 — the partial state of the SPEARMAN
 *                            aggregate (tg_plan_set_aggregate_partial), which merges across ranks by addition
 * Equal keys always meet on one rank, so ties share the global minimum rank exactly as on one GPU. tg_rank_abort drops
 * the session. On one GPU tg_plan_execute runs the same stages back to back.
 */
TG_API tg_status tg_rank_begin(tg_engine* eng, const char* table, const char* column_x, const char* column_y, int64_t* n_pairs);
TG_API tg_status tg_rank_local_sort(tg_engine* eng);
TG_API int32_t tg_rank_sample(tg_engine* eng, int32_t n_samples, uint64_t* keys);
TG_API tg_status tg_rank_split(tg_engine* eng, const uint64_t* splitters, int32_t n_parts, int64_t* counts);
TG_API tg_status tg_rank_send_buffers(tg_engine* eng, const void** keys, const void** payload, int32_t* payload_bytes);
TG_API tg_status tg_rank_recv_buffers(tg_engine* eng, int64_t n_recv, void** keys, void** payload);
TG_API tg_status tg_rank_recv_commit(tg_engine* eng, int64_t n_recv);
TG_API tg_status tg_rank_finish_x(tg_engine* eng, uint64_t rank_base);
TG_API tg_status tg_rank_finish_y(tg_engine* eng, uint64_t rank_base, double center, uint64_t* n_out, double* sums5);
TG_API tg_status tg_rank_abort(tg_engine* eng);
/* The exchange between tg_rank_begin / tg_rank_finish_x / tg_rank_finish_y done by the library itself (needs tg_comm_init):
 * samples all-gathered over NCCL, splitters, then the session's (key, payload) pairs are PUSHED to the ranks that own
 * their key ranges by the partition's scatter kernel — NVLink peer stores into IPC-mapped receive buffers, no local
 * pre-sort and no separate all-to-all. Returns the rows this rank now holds, the number of keys on the lower ranks
 * (rank_base of the finish calls) and the global pair count. *done = 0: peer mapping is unavailable, nothing happened;
 * run tg_rank_local_sort / _sample / _split and an all-to-all of your own instead. */
TG_API tg_status tg_rank_exchange(tg_engine* eng, int64_t* n_recv, uint64_t* rank_base, uint64_t* total, int32_t* done);
/* Installs a partial state computed outside tg_plan_execute_partial for aggregate i (kind 10 SPEARMAN only): u[0] = pair
 * count, f[0] = f[1] = center, f[2..6] = the five sums. Call it after tg_plan_execute_partial, before the exchange. */
TG_API tg_status tg_plan_set_aggregate_partial(tg_plan* plan, int32_t i, const uint64_t* u8, const double* f8);

/* The sketch behind a tg_plan_add_kll / quantile slot as KllSketch's own fields (kll_sketch.rs:142-160): count / min /
 * max come with tg_plan_analyzer_result; this returns the compactor stack. level < 0: the number of levels; otherwise
 * the items of that level (each standing for 2^level values, ascending) are copied into items[cap] and the level's item
 * count is returned. A shim can rebuild a reference-side KllSketch from it, or merge per level like KllSketch::merge
 * (:327-366). */
TG_API int32_t tg_plan_kll_levels(const tg_plan* plan, int32_t slot, int32_t level, double* items, int32_t cap);

/* Two-phase histogram over row shards (analyzers/advanced/histogram.rs:184-290 derives the bucket bounds from the
 * table-wide MIN / MAX, so shards that saw different ranges cannot add their counts). After the shards' partials were
 * merged (tg_plan_partial_merge / tg_plan_exchange_and_finalize), tg_plan_histogram_pending lists the HIST aggregates
 * whose shards disagreed on [min, max] (returns their number; fills up to `cap` indices). For each of them every rank
 * calls tg_plan_histogram_rebucket, which counts ITS shard `table_name` against the merged (global) min / max of the
 * plan's NUM aggregate into counts[n_buckets]; the host layer sums the counts over the ranks (a u64 all-reduce) and
 * every rank installs the sums and calls tg_plan_finalize again. */
TG_API int32_t tg_plan_histogram_pending(const tg_plan* plan, int32_t* agg_indices, int32_t cap);
TG_API tg_status tg_plan_histogram_rebucket(tg_engine* eng, tg_plan* plan, const char* table_name, int32_t agg_index,
                                            uint64_t* counts, int32_t n_buckets);
TG_API tg_status tg_plan_histogram_install(tg_plan* plan, int32_t agg_index, const uint64_t* counts, int32_t n_buckets);

/* Multi-GPU shuffle, step 3: aggregate i (kind 6 DISTINCT or 7 FK) reads its keys from `table_name` — the table
 * holding this rank's hash-shuffled shard (tg_table_partition_keys + all-to-all + tg_table_adopt_device) — instead
 * of the plan's table; which = 0: the DISTINCT table / the FK child table, 1: the FK parent table. NULL or ""
 * removes the redirection. Shards are hash-disjoint, so tg_plan_partial_merge adds their states exactly. */
TG_API tg_status tg_plan_redirect_aggregate(tg_plan* plan, int32_t i, int32_t which, const char* table_name);

TG_API tg_status tg_plan_result(const tg_plan* plan, int32_t slot, tg_result* out);
TG_API tg_status tg_plan_analyzer_result(const tg_plan* plan, int32_t slot, tg_analyzer_result* out);
/* Map-valued metrics (KLL, grouped completeness, stddev): entry i of slot */
TG_API int32_t tg_plan_map_size(const tg_plan* plan, int32_t slot);
TG_API tg_status tg_plan_map_entry(const tg_plan* plan, int32_t slot, int32_t i, const char** key,
                                   double* value);

/* The analyzer slot's *State struct as serde_json text — what IncrementalAnalysisRunner hands to a StateStore
 * (analyzers/incremental/runner.rs:72-80; FileSystemStateStore writes it to {partition}/{analyzer}.json,
 * state_store.rs:153-176), so GPU-computed partitions can be mixed with CPU-computed ones (SURVEY §8f.4). Writes
 * NUL-terminated into buf, returns the needed length (0: this slot has no JSON state, e.g. KLL / grouped / Spearman;
 * negative: -tg_status). */
TG_API int32_t tg_plan_analyzer_state_json(const tg_plan* plan, int32_t slot, char* buf, int32_t cap);

/* timings of the last execute, milliseconds (SURVEY §5 metrics row): h2d, scan kernels, total */
typedef struct {
    double gpu_ms;        /* CUDA-event time of all kernels of the last execute */
    double scan_ms;       /* fused numeric scan kernel only */
    double string_ms;
    double hash_ms;
    double sketch_ms;
    uint64_t bytes_scanned; /* algorithmic bytes (SURVEY §8d) of the last execute */
    uint64_t launches;
} tg_exec_stats;
TG_API tg_status tg_plan_exec_stats(const tg_plan* plan, tg_exec_stats* out);

/* Test hook (not part of the reference-facing surface): the hand-written sm_100a radix sort behind K6 (Spearman's
 * RANK() OVER (ORDER BY ..), analyzers/advanced/correlation.rs:334-350) and K4 on its own — `n` host keys are sorted
 * (stably) by the key bits [begin_bit, begin_bit + 8 * n_passes); out_index receives each sorted key's original
 * position. The parity tests compare it with numpy's stable argsort. */
TG_API tg_status tg_debug_sort_pairs(tg_engine* eng, const uint64_t* keys, int64_t n, int32_t begin_bit, int32_t n_passes,
                                     uint64_t* out_keys, uint32_t* out_index);

/* -------------------------------------------------- host-side helpers ---- */
/* These restate O(1) reference host logic so the shim and tests can call it without a GPU. */

/* Assertion::evaluate (constraints/assertion.rs:48-61) */
TG_API int32_t tg_assertion_evaluate(tg_assertion a, double value);
/* Assertion::description (assertion.rs:64-75); writes NUL-terminated into buf, returns needed length */
TG_API int32_t tg_assertion_description(tg_assertion a, char* buf, int32_t cap);
/* LogicalOperator::evaluate (core/logical.rs:69-89) */
TG_API int32_t tg_logical_evaluate(int32_t op, int32_t n, const uint8_t* results, int32_t n_results);
/* SqlSecurity::validate_identifier (security.rs:89-137) */
TG_API tg_status tg_validate_identifier(const char* identifier);
/* SqlSecurity::validate_regex_pattern (security.rs:152-183) + our DFA grammar check */
TG_API tg_status tg_validate_regex_pattern(const char* pattern);
/* custom_sql.rs:100-190 validate_sql_expression */
TG_API tg_status tg_validate_sql_expression(const char* expression);
/* FormatType::get_pattern (constraints/format.rs:217-307) */
TG_API const char* tg_format_pattern(int32_t format_kind, const char* arg, int32_t flag);
/* Host DFA matcher used ONLY to unit-test the regex compiler without a GPU (the product path runs the
 * same table on the device): returns 1/0 match of `pattern` (search semantics of `~`) on bytes. */
TG_API int32_t tg_regex_host_match(const char* pattern, int32_t case_insensitive, const uint8_t* s,
                                   int64_t len, int32_t* out_match);
/* Size of the minimised byte DFA a pattern compiles to (states incl. DEAD / MATCH, byte classes): what the string
 * kernel's shared-memory table holds. */
TG_API int32_t tg_regex_dfa_size(const char* pattern, int32_t case_insensitive, uint32_t* n_states, uint32_t* n_classes);
/* serde_json (ryu) rendering of an f64, as in the persisted analyzer states; returns needed length */
TG_API int32_t tg_format_f64_json(double v, char* buf, int32_t cap);
/* Rust `{}` Display of f64, for message parity; returns needed length */
TG_API int32_t tg_format_f64(double v, char* buf, int32_t cap);

#ifdef __cplusplus
}
#endif
#endif /* TERMGPU_H */
