// Plan = fused form of a Check / ValidationSuite / AnalysisRunner.
//   slots      : one per constraint or analyzer the caller added (what the reference evaluates with
//                one SQL query each, core/suite.rs:84-100)
//   aggregates : the de-duplicated device work the slots need; each aggregate has a partial state that
//                merges across row shards (GPUs) like AnalyzerState::merge (analyzers/traits.rs:154-179)
#pragma once
#include <functional>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "common.hpp"
#include "sqlexpr.hpp"

namespace tg {

enum AggKind : int32_t {
    A_ROWS = 0,      // COUNT(*)                       u0 rows
    A_VALID = 1,     // COUNT(c)                       u0 rows u1 non-null
    A_NUM = 2,       // numeric moments/min/max/sum    u0 n u1 isum u2 imin u3 imax u4 is_i64 | f0 K f1 Σd f2 Σd² f3 min f4 max f5 Σx
    A_PAIR = 3,      // pairwise-complete co-moments   u0 n | f0 Kx f1 Ky f2 Σdx f3 Σdy f4 Σdx² f5 Σdy² f6 Σdxdy
    A_PRED = 4,      // COUNT(CASE WHEN p THEN 1 END)  u0 true u1 div0 u2 rows
    A_REGEX = 5,     // c ~ 'pat'                      u0 matches(non-null) u1 nulls u2 rows
    A_DISTINCT = 6,  // COUNT(DISTINCT ..)/GROUP BY    u0 rows u1 distinct(non-null keys) u2 singleton groups u3 rows-with-any-null u4 null-group-rows u5 distinct-with-null-as-value
    A_FK = 7,        // LEFT JOIN anti-count           u0 violations u1 distinct violations u2 null child rows ; blob = example keys
    A_KLL = 8,       // blob = sketch
    A_GROUPED = 9,   // blob = group table
    A_SPEARMAN = 10, // same layout as A_PAIR over min-ranks
    A_LENGTH = 11,   // COUNT(CASE WHEN lo <= LENGTH(c) <= hi ..)  u0 matching non-null rows u1 nulls u2 rows
    A_HIST = 12,     // equal-width histogram over [min, max] of the column's NUM aggregate: f0 min f1 max u0 is_i64 u7 pending (shards disagreed on the range) ; blob = bucket counts
};

struct RowMask;

struct Agg {
    AggKind kind;
    std::string key;                 // de-duplication key
    std::vector<std::string> cols;   // for A_FK: child table, child col, parent table, parent col
    std::string text;                // predicate / regex pattern
    int32_t flags = 0;               // regex: bit0 case-insensitive, bit1 trim ; distinct: see hash job ; grouped: bit1 = value histogram
                                     // (keys print as CAST(.. AS VARCHAR): booleans true / false, no floating point)
    int32_t iparam = 0;              // KLL k / FK max examples / grouped max_groups
    int64_t lo = 0, hi = 0;          // A_LENGTH: inclusive character-count range
    ExprP expr;                      // parsed predicate
    // multi-GPU shuffle: read this aggregate's keys from another registered table (the hash-shuffled shard) instead
    // of the plan's table; [0] = the table of a DISTINCT aggregate or the child table of an FK, [1] = the FK parent
    std::string redirect[2];
    // some slot requested its row verdicts (tg_plan_request_row_mask): the kernels of this aggregate also store one word per 32
    // rows to `bits` (device, held by execute_partial for the duration of one execute). Not part of the de-duplication key.
    bool row_bits = false;
    uint32_t* bits = nullptr;
    // key-level row verdicts some slot requested (tg_plan_request_key_rows): bit k = tg_key_rows_kind k. The hash job of this
    // aggregate builds key_mask[k] for the execute's rows; the slots take them over. Not part of the de-duplication key.
    uint8_t key_rows = 0;
    std::shared_ptr<RowMask> key_mask[3];
    // construction-time problem the reference only reports when the constraint is evaluated
    tg_status ctor_err = TG_OK;
    std::string ctor_err_msg;
    // ---- bind status of the last execute ----
    tg_status err = TG_OK;
    std::string err_msg;
    // DataFusion result typing of the (first) column's aggregates: bit 0: MIN / MAX / APPROX_PERCENTILE_CONT keep a type that
    // is neither Int64 nor Float64 (Int8..Int32, UInt*, Float32); bit 1: SUM is UInt64 (unsigned columns). narrow_name: that type
    int32_t narrow = 0;
    const char* narrow_name = "";
    // ---- partial state ----
    uint64_t u[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    double f[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    std::vector<uint8_t> blob;
    void reset_state() {
        for (auto& x : u) x = 0;
        for (auto& x : f) x = 0;
        blob.clear();
        err = ctor_err;
        err_msg = ctor_err_msg;
        narrow = 0;
        for (auto& m : key_mask) m.reset();
    }
};

enum SlotKind : int32_t {
    SL_COMPLETENESS,
    SL_SIZE,
    SL_STAT,
    SL_MULTISTAT,
    SL_FORMAT,
    SL_UNIQ,
    SL_CORR,
    SL_SQL,
    SL_FK,
    SL_ANALYZER,
    SL_KLL,
    SL_GROUPED,
    SL_LENGTH,
    SL_CONTAINMENT,
    SL_NON_NEGATIVE,
    SL_APPROX_DISTINCT,
    SL_DATA_TYPE,
    SL_COLUMN_COUNT,
    SL_HISTOGRAM,
    SL_QUANTILE,
    SL_VALUE_HIST,
};

// One slot's row verdicts as an Arrow Boolean array in device memory (engine.cu build_row_masks): values bit i = row i is in
// the metric's numerator, validity bit i = row i is in its denominator (validity null: every row). Shared between the slot and
// the arrays exported from it; the last owner hands the buffers back to the engine through `give_back`.
struct RowMask {
    int64_t n_rows = 0, null_count = 0;
    uint8_t* values = nullptr;
    uint8_t* validity = nullptr;
    size_t bytes = 0;  // capacity of each buffer
    int device = 0;
    std::function<void(uint8_t*, size_t)> give_back;
    ~RowMask() {
        if (give_back) {
            give_back(values, bytes);
            if (validity) give_back(validity, bytes);
        }
    }
};

struct StatReq {
    int32_t kind;
    double percentile;
    tg_assertion assertion;
    int agg_kll = -1;
};

struct Slot {
    SlotKind kind;
    // parameters
    std::vector<std::string> columns;
    double threshold = 1.0;
    int32_t op = TG_OP_ALL, op_n = 0;
    tg_assertion assertion{0, 0, 0};
    std::vector<StatReq> stats;
    int32_t sub_kind = 0;      // format kind / uniqueness kind / correlation kind / analyzer kind
    std::string arg;           // format arg / SQL expression
    bool has_arg = false;
    int32_t flag = 0;
    tg_format_options fopt{1, 0, 1};
    std::string pattern;       // resolved regex
    std::string hint;
    bool has_hint = false;
    int32_t null_handling = 0;
    int32_t allow_nulls = 0, max_examples = 100;
    std::vector<double> quantiles;
    int32_t k = 0;
    int32_t max_groups = 10000, include_overall = 1;
    // aggregates feeding this slot (meaning depends on kind)
    std::vector<int> aggs;
    // results
    std::string name;
    int32_t status = TG_SKIPPED;
    bool has_metric = false;
    double metric = 0;
    bool has_message = false;
    std::string message;
    tg_analyzer_result ares{};
    std::string metric_key;
    std::vector<std::pair<std::string, double>> map;
    // row verdicts: requested before execute; the mask (or the reason there is none) of the last execute since the request
    // key-level row verdicts (uniqueness and foreign-key slots): bit k of key_rows_requested = tg_key_rows_kind k; they share
    // mask_built / mask_err with the row mask, which these slots never have
    bool mask_requested = false, mask_built = false;
    std::shared_ptr<RowMask> mask;
    uint8_t key_rows_requested = 0;
    std::shared_ptr<RowMask> key_rows[3];
    tg_status mask_err = TG_OK;
    std::string mask_err_msg;
};

// slot kinds whose row verdicts can be exported; false for the others (and for completeness over several columns)
bool slot_has_row_mask(const Slot& s);

struct Plan {
    std::vector<Agg> aggs;
    std::vector<Slot> slots;
    tg_exec_stats stats{};
    bool executed = false;

    int add_agg(Agg a);  // de-duplicates on key
    void reset_partials();
    size_t partial_size() const;
    void partial_export(uint8_t* buf) const;
    void partial_merge(const uint8_t* buf, size_t n);  // merge another shard's partials into ours
    void merge_state(int i, tg_status err, const std::string& emsg, const uint64_t* u, const double* f, const std::vector<uint8_t>& blob);
    void finalize();                                    // slots <- aggregates
    std::vector<int> histogram_pending() const;         // HIST aggregates waiting for the second (global-range) phase
    void histogram_install(int agg_id, const uint64_t* counts, int nb);
};

// slot constructors (validate like the reference constructors do; throw Error)
int plan_add_completeness(Plan& p, const std::vector<std::string>& cols, double threshold, int op, int op_n);
int plan_add_size(Plan& p, tg_assertion a);
int plan_add_statistic(Plan& p, const std::string& col, int stat, double pct, tg_assertion a);
int plan_add_multi_statistic(Plan& p, const std::string& col, const std::vector<StatReq>& stats);
int plan_add_format(Plan& p, const std::string& col, int kind, const char* arg, int flag, double threshold,
                    tg_format_options opt);
int plan_add_uniqueness(Plan& p, const std::vector<std::string>& cols, int kind, double threshold,
                        tg_assertion a, int null_handling);
int plan_add_correlation(Plan& p, const std::string& c1, const std::string& c2, int kind, tg_assertion a);
int plan_add_custom_sql(Plan& p, const std::string& expr, const char* hint);
int plan_add_foreign_key(Plan& p, const std::string& child, const std::string& parent, int allow_nulls,
                         int max_examples);
int plan_add_analyzer(Plan& p, int kind, const char* col, const char* col2, const char* expr);
int plan_add_kll(Plan& p, const std::string& col, int k, const std::vector<double>& q);
int plan_add_length(Plan& p, const std::string& col, int kind, int64_t a, int64_t b);
int plan_add_containment(Plan& p, const std::string& col, const std::vector<std::string>& allowed);
int plan_add_non_negative(Plan& p, const std::string& col);
int plan_add_approx_count_distinct(Plan& p, const std::string& col, tg_assertion a);
int plan_add_data_type(Plan& p, const std::string& col, int data_type, double threshold);
int plan_add_column_count(Plan& p, tg_assertion a);
int plan_add_histogram(Plan& p, const std::string& col, int num_buckets);
int plan_add_quantile(Plan& p, const std::string& col, int mode, const std::vector<double>& quantiles,
                      const std::vector<tg_assertion>& assertions, int strict);
// HistogramConstraint (constraints/histogram.rs:208-244): value frequencies of one column, as a grouped count of the column by itself
int plan_add_value_histogram(Plan& p, const std::string& col);
// marks a slot's row verdicts for the next execute (TG_ERR_UNSUPPORTED for a kind without them, TG_ERR_INVALID_ARG out of range)
void plan_request_row_mask(Plan& p, int slot);
// marks one kind of a uniqueness / foreign-key slot's key-level row verdicts for the next execute (TG_ERR_UNSUPPORTED for other
// slot kinds, TG_ERR_INVALID_ARG for a kind the slot has not or an index out of range)
void plan_request_key_rows(Plan& p, int slot, int kind);
// the slot a key-level verdict of `kind` can be exported from (the same errors as plan_request_key_rows)
const Slot& key_rows_slot(const Plan& p, int slot, int kind);
int plan_add_grouped_completeness(Plan& p, const std::string& col, const std::vector<std::string>& groups,
                                  int max_groups, int include_overall);

// serde_json text of an analyzer slot's *State struct, as IncrementalAnalysisRunner / FileSystemStateStore persist it
// (analyzers/incremental/runner.rs:72-80, state_store.rs:153-176); empty string when the slot has no such state
std::string analyzer_state_json(const Plan& p, int slot);

// KLL sketch blob helpers (kll_host.cpp)
struct KllHost;
void kll_blob_merge(std::vector<uint8_t>& into, const std::vector<uint8_t>& other);
bool kll_blob_query(const std::vector<uint8_t>& blob, double phi, double* out);
void kll_blob_summary(const std::vector<uint8_t>& blob, uint64_t* n, double* mn, double* mx);
int kll_blob_levels(const std::vector<uint8_t>& blob, std::vector<std::vector<double>>& levels, uint64_t* k);

// grouped table blob helpers (plan.cpp)
void grouped_blob_merge(std::vector<uint8_t>& into, const std::vector<uint8_t>& other);

}  // namespace tg
