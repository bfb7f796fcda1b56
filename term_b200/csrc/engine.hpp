// Engine / table / column objects behind the C ABI. Device memory layout (DESIGN.md §3):
// every column is ONE contiguous Arrow-layout buffer set in HBM (values, validity bitmap LSB-first,
// int32 offsets for Utf8), 256-byte aligned, zero padded to a multiple of 256 bytes so TMA bulk copies
// and 128-bit loads may over-read the tail.
#pragma once
#include <cuda_runtime.h>

#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "common.hpp"
#include "plan.hpp"
#include "scan_defs.h"

namespace tg {

#define TG_CUDA(expr)                                                                                   \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess)                                                                          \
            throw ::tg::Error(TG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));         \
    } while (0)

struct Engine;
struct RankSession;  // ranks.cu: state of a Spearman evaluation between its stages

struct DevBuf {
    uint8_t* p = nullptr;
    size_t cap = 0;
    bool owned = true;
};

struct Column {
    std::string name;
    int32_t dtype = 0;
    int64_t n_rows = 0;
    DevBuf values;      // fixed width: n*w bytes; Utf8: value bytes; Bool: bit-packed
    DevBuf offsets;     // Utf8: (n+1) int32
    DevBuf validity;    // p == nullptr: no nulls so far
    int64_t value_bytes = 0;
    int64_t null_count = 0;
    uint8_t tail_byte = 0;   // host mirror of the last, partially filled validity byte
    uint8_t tail_vbyte = 0;  // same for bit-packed Bool values
    int32_t last_offset = 0;
    bool pivot_set = false;       // a finite, valid element of the column was found
    double pivot = 0.0;           // shift K of the moment sums (== (double)ipivot for Int64 columns)
    int64_t ipivot = 0;
    bool adopted = false;
    // Int32 / Float32 columns: the exact 8-byte (Int64 / Float64) shadow the numeric aggregates, predicates, sketches and
    // rank sorts read (numeric_view, engine.cu): built on the device on first use, rebuilt when rows were appended since
    std::unique_ptr<Column> wide;
    // Arrow type the column was delivered as when it is not the stored one (Int8 .. UInt64 / Date / Timestamp / Time /
    // Duration columns are stored as Int32 / Int64): DataFusion types MIN / MAX (and SUM of unsigned columns) after it
    const char* src_type = nullptr;  // static string ("UInt16", "Date32", "Timestamp(Microsecond, None)", ..)
    bool src_unsigned = false;
    bool temporal = false;           // comparisons / completeness / uniqueness / grouping only: no numeric aggregates
    char temporal_unit = 0;          // 'D' days (Date32), 's' / 'm' / 'u' / 'n' (Date64 is 'm', Timestamp by unit); 0: times, durations
    int elem_bytes() const {
        switch (dtype) {
            case TG_INT64: case TG_FLOAT64: return 8;
            case TG_INT32: case TG_FLOAT32: return 4;
            default: return 0;
        }
    }
};

struct Table {
    Engine* eng = nullptr;
    std::string name;
    std::vector<std::unique_ptr<Column>> cols;
    int64_t n_rows = 0;
    Column* find(const std::string& n) {
        for (auto& c : cols)
            if (c->name == n) return c.get();
        return nullptr;
    }
    std::string valid_fields() const {
        std::string s;
        for (size_t i = 0; i < cols.size(); ++i) {
            if (i) s += ", ";
            s += name + "." + cols[i]->name;
        }
        return s;
    }
};

// Fused multi-GPU step of a scan-only plan (engine.cu execute_exchange_fused): the aggregates' partial states are
// assembled on the device behind the scan instead of on the host.
struct DevAggRec {  // what travels between the ranks per aggregate: the partial state of plan.hpp's Agg
    uint64_t kind, err;
    uint64_t u[8];
    double f[8];
};
struct ScanOpMeta {  // how scan_states_kernel turns one ScanAggOut record into a DevAggRec
    int32_t unit_kind, agg;
    double pivot0, pivot1;
    uint64_t n_rows;
};
struct FusedScan {
    DevAggRec* d_states = nullptr;  // [n_aggs], zeroed; written by scan_states_kernel after every pass
    ScanOpMeta* d_metas = nullptr;  // [n_aggs] device
    ScanOpMeta* h_metas = nullptr;  // [n_aggs] pinned
    int n_metas = 0;
    std::vector<uint8_t> from_device;          // per aggregate: its state comes from d_states
    std::vector<std::pair<int, int>> folds;    // (VALID aggregate, NUM aggregate whose count it takes)
    int launches = 0;
};

// peer mailboxes of the multi-GPU partial-state exchange (mailbox.cu)
constexpr int MAILBOX_MAX_WORLD = 16;
struct MailboxPeers {
    uint8_t* p[MAILBOX_MAX_WORLD];
};
struct Mailbox {
    int world = 0, rank = 0;
    size_t slot_bytes = 0, bytes = 0;
    uint8_t* local = nullptr;     // this rank's mailbox (device)
    MailboxPeers peers{};         // every rank's mailbox as seen from this device (IPC-mapped)
    uint8_t* d_stage = nullptr;   // this rank's outgoing blob (device) + timeout flag
    uint8_t* h_stage = nullptr;   // pinned
    uint8_t* h_all = nullptr;     // pinned landing area of a collected step
    unsigned long long seq = 0;
    bool open = false;
};

struct Engine {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;       // kernels
    cudaStream_t copy_stream = nullptr;  // H2D staging
    cudaEvent_t ev[8] = {};
    uint8_t* pinned[2] = {nullptr, nullptr};
    cudaEvent_t pinned_free[2] = {};
    size_t pinned_bytes = 0;
    int pinned_next = 0;
    std::map<std::string, std::unique_ptr<Table>> tables;
    std::mutex mu;
    uint64_t launches = 0;
    // scratch
    uint8_t* d_scratch = nullptr;
    size_t scratch_cap = 0;
    uint8_t* h_scratch = nullptr;  // pinned
    size_t h_scratch_cap = 0;
    uint8_t* d_shuffle = nullptr;  // keys grouped by destination rank (multi-GPU shuffle), grow-only
    size_t shuffle_cap = 0;

    // recycled device blocks of dropped tables, by exact capacity
    std::map<size_t, std::vector<uint8_t*>> free_blocks;
    size_t cached_bytes = 0;
    size_t cache_limit = (size_t)48 << 30;
    uint8_t* dev_alloc(size_t bytes);
    void dev_free(uint8_t* p, size_t bytes);
    void dev_trim();

    // side streams: independent bucket pipelines of the partitioned hash jobs run concurrently on them
    cudaStream_t side[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t side_ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    void ensure_side_streams();
    Mailbox mailbox;
    RankSession* rank_session = nullptr;
    int64_t rank_cap_hint = 0;  // largest rank arena so far: later arenas take that size and hit the device-block cache
    // NCCL communicator of the hash shuffle behind the C ABI (comm.cpp; libnccl bound at run time)
    void* comm = nullptr;
    int comm_world = 0, comm_rank = 0;
    uint8_t* d_comm_counts = nullptr;
    uint8_t* d_comm_samples = nullptr;
    void* push = nullptr;          // comm.cpp PushState: IPC-mapped receive buffers of the push shuffle
    uint64_t comm_bytes_sent = 0;  // bytes this rank sent to OTHER ranks through tg_table_shuffle_* since creation
    FusedScan* fused = nullptr;  // non-null while execute_exchange_fused runs the scan jobs
    uint8_t* d_aux = nullptr;  // small grow-only device block for result post-processing (group keys, ..)
    size_t aux_cap = 0;
    uint8_t* aux(size_t bytes);
    uint8_t* scratch(size_t bytes);
    uint8_t* host_scratch(size_t bytes);
    void dev_reserve(DevBuf& b, size_t need, size_t keep_bytes);
    // staged through the pinned ring unless src is pinned; queued on `s` (nullptr: copy_stream)
    void h2d(void* dst, const void* src, size_t bytes, cudaStream_t s = nullptr);
    void sync_copies();
    // device blocks still read by work queued on copy_stream (Parquet staging): released by the next sync_copies()
    std::vector<std::pair<uint8_t*, size_t>> deferred_free;
};

// the column itself when it is Int64 / Float64, the widened shadow of an Int32 / Float32 column, nullptr for other types
Column* numeric_view(Engine& e, Column* c);
void column_free(Engine& e, Column& c);

// One append call (tg_table_append_*): holds the engine's lock and makes the call all or nothing. A call that throws
// leaves the table as it was: every column it touched gets back its rows, byte count, NULL count, tail mirrors, pivot and
// declared type, a validity bitmap the call created is freed, the columns it created are dropped. Capacity the call grew
// is kept (it lies past the column's end). A successful call pays nothing for this but the record of the columns it touched.
class AppendTxn {
  public:
    explicit AppendTxn(Table& t);
    ~AppendTxn();
    // the column to append to (created with `dtype` when missing); adopted device columns are refused
    Column& column(const std::string& name, int32_t dtype);
    // the call succeeded: the table's row count becomes the largest of its touched columns
    void commit();
    Engine& e;
    Table& t;

  private:
    struct Saved {
        Column* c;
        int64_t n_rows, value_bytes, null_count;
        int32_t last_offset;
        uint8_t tail_byte, tail_vbyte;
        bool pivot_set, had_validity;
        double pivot;
        int64_t ipivot;
        const char* src_type;
        bool src_unsigned, temporal;
        char temporal_unit;
    };
    std::lock_guard<std::mutex> g;
    size_t n_cols;
    int64_t n_rows;
    std::vector<Saved> saved;
    bool committed = false;
};

// tables.cu helpers shared with the Parquet path (parquet.cu)
Column* table_get_or_add(Table& t, const std::string& name, int32_t dtype);
void set_pivot_host(Column& c, int32_t dtype, int64_t n, const void* values, const uint8_t* validity, int64_t bit_offset);
void append_validity(Engine& e, Column& c, int64_t have, const uint8_t* validity, int64_t bit_offset, int64_t n);
// device-side counterparts for the CSV path (csv.cu): `words` = a chunk-relative device bitmap of n rows (bit r of word r / 32),
// last64 = its bits of rows n - 64 .. n - 1 (bit k: row n - 64 + k) read back from the device, zeros = its clear bits
void append_validity_device(Engine& e, Column& c, int64_t have, const uint32_t* words, int64_t n, int64_t zeros, uint64_t last64);
void append_bits_device(Engine& e, DevBuf& buf, uint8_t& tail, int64_t have, const uint32_t* words, int64_t n, uint64_t last64);
// table_set_column_arrow_type without the engine's lock (the caller holds it)
void declare_arrow_type(Column& c, const std::string& fmt);

// jobs (each fills the partial state of the aggregates it owns)
void exec_scan_jobs(Engine& e, Table& t, Plan& p, const std::vector<int>& agg_ids);   // engine.cu + scan.cu
void exec_string_jobs(Engine& e, Table& t, Plan& p, const std::vector<int>& agg_ids); // strings.cu
void exec_length_jobs(Engine& e, Table& t, Plan& p, const std::vector<int>& agg_ids); // strings.cu
void exec_distinct_job(Engine& e, Table& t, Plan& p, int agg_id);                     // hashing.cu
void exec_fk_job(Engine& e, Plan& p, int agg_id);                                     // hashing.cu
void exec_kll_jobs(Engine& e, Table& t, Plan& p, const std::vector<int>& agg_ids);  // sketch.cu
void exec_grouped_jobs(Engine& e, Table& t, Plan& p, const std::vector<int>& agg_ids); // grouped.cu (all groupings of a plan in one pass)
void exec_spearman_job(Engine& e, Table& t, Plan& p, int agg_id);                     // ranks.cu
void exec_hist_job(Engine& e, Table& t, Plan& p, int agg_id);                         // hist.cu
// ranks.cu: the stages of the (distributed) rank computation behind tg_rank_*
void rank_session_destroy(Engine& e);
int64_t rank_begin(Engine& e, const std::string& table, const std::string& cx, const std::string& cy);
void rank_local_sort(Engine& e);
int32_t rank_sample(Engine& e, int32_t m, uint64_t* out);
void rank_split(Engine& e, const uint64_t* splitters, int32_t n_parts, int64_t* counts);
void rank_send_buffers(Engine& e, const void** keys, const void** payload, int32_t* payload_bytes);
void rank_recv_buffers(Engine& e, int64_t n_recv, void** keys, void** payload);
void rank_recv_commit(Engine& e, int64_t n_recv);
void rank_finish_x(Engine& e, uint64_t rank_base);
void rank_finish_y(Engine& e, uint64_t rank_base, double K, uint64_t* n_out, double* sums);
void rank_abort(Engine& e);
void rank_current_unlocked(Engine& e, const uint64_t** keys, const void** payload, int* pay_bytes, int64_t* n);
int32_t rank_sample_unlocked(Engine& e, int32_t m, uint64_t* out);
void rank_adopt_received_unlocked(Engine& e, uint64_t* keys, void* payload, int64_t n_recv);
int rank_phase_unlocked(Engine& e);
void hist_rebucket(Engine& e, Table* t, Plan& p, int agg_id, uint64_t* counts, int nb); // hist.cu (two-phase multi-GPU histogram)

void execute_partial(Engine& e, Plan& p, const std::string& table_name);
bool execute_exchange_fused(Engine& e, Plan& p, const std::string& table_name);  // false: not applicable, nothing done

// mailbox.cu
void mailbox_create(Engine& e, int world, int rank, size_t slot_bytes, void* handle_out /* 64 bytes */);
void mailbox_open(Engine& e, const void* handles /* world x 64 bytes */);
void mailbox_destroy(Engine& e);
bool mailbox_exchange(Engine& e, const uint8_t* blob, size_t n, std::vector<std::vector<uint8_t>>& out);
void mailbox_exchange_device(Engine& e, size_t payload_bytes, std::vector<std::vector<uint8_t>>& out);

// comm.cpp
void comm_unique_id(void* id128);
void comm_init(Engine& e, const void* id128, int world, int rank);
void comm_destroy(Engine& e);
int64_t comm_shuffle_column(Engine& e, const std::string& table, const std::string& column, const std::string& shard_name, bool allow_range);
bool comm_rank_exchange(Engine& e, int64_t* n_recv, uint64_t* rank_base, uint64_t* total);  // false: push exchange unavailable
int64_t comm_shuffle_fingerprints(Engine& e, const std::string& table, const std::vector<std::string>& columns, const std::string& shard_name);

// scan.cu
size_t scan_smem_bytes(const ScanParams& P);
cudaError_t scan_launch(const ScanParams& P, int grid, ScanAggOut* d_out, cudaStream_t stream);

}  // namespace tg
