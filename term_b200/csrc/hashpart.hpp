// Radix-partitioned hash jobs for large Int64 / Float64 key columns (hashpart.cu).
#pragma once
#include <cstdint>
#include <vector>

#include "engine.hpp"

namespace tg {

// key-level row verdicts (hash_common.cuh): a counting path given R (not nullptr) also inserts every key it sees a second
// time into R; a foreign-key path given `orphan_rows` also writes the child rows whose key it found without a parent
struct RepTab;
struct VerdictOut;
void rep_reset(Engine& e, const RepTab& R);              // empties R before a counting attempt
void rep_mark(Engine& e, const RepTab& R, uint64_t key);  // a key the path counted apart occurs twice or more
void fk_orphan_rows64(Engine& e, const Column& child, int64_t nc, const unsigned long long* vkeys, uint64_t vmask, int shift,
                      bool special_orphan, const VerdictOut& out, int& launches);

struct Distinct64Result {
    uint64_t distinct = 0;   // distinct non-null keys
    uint64_t dup_keys = 0;   // keys that occur at least twice
    uint64_t nulls = 0;      // NULL rows
};
// COUNT(DISTINCT c) / GROUP BY c HAVING COUNT(*) = 1 over a single 64-bit key column. Returns false when a bucket
// table overflowed (pathologically skewed hash): the caller falls back to the single-table path.
bool distinct64_partitioned(Engine& e, const Column& c, int64_t n, Distinct64Result& r, int& launches, const RepTab* R = nullptr);
size_t distinct64_min_rows();
// The same counts for sparse keys without a global atomic (hashsort.cu): hashes of the valid keys, two or three radix passes
// over their low bits, shared-memory de-duplication of the contiguous hash buckets. Returns false (nothing counted) on a
// hot key / skewed bucket or for n >= 2^30: the caller takes the partitioned path.
bool distinct64_sorted(Engine& e, const Column& c, int64_t n, Distinct64Result& r, int& launches, const RepTab* R = nullptr);
// Dense Int64 key range (max - min < 2^28 and < 32 n): exact bitmap counting, no partitioning. Returns false when
// the column does not qualify (nothing is counted then).
bool distinct64_dense(Engine& e, const Column& c, int64_t n, bool need_singles, Distinct64Result& r, int& launches,
                      const RepTab* R = nullptr);

struct Fk64Result {
    uint64_t violations = 0;           // child rows without a parent (NULL children included when not allowed)
    uint64_t distinct_violations = 0;  // distinct orphan keys
    uint64_t null_children = 0;
    std::vector<uint64_t> example_keys;  // up to max_examples distinct orphan keys (raw 64-bit values)
};
bool fk64_partitioned(Engine& e, const Column& child, int64_t nc, const Column& parent, int64_t np, int allow_nulls,
                      int max_examples, Fk64Result& r, int& launches, const VerdictOut* orphan_rows = nullptr);

bool fk64_dense(Engine& e, const Column& child, int64_t nc, const Column& parent, int64_t np, int allow_nulls, int max_examples,
                Fk64Result& r, int& launches, const VerdictOut* orphan_rows = nullptr);

// Multi-GPU shuffle, step 1 (SURVEY §8e): the valid keys of a column grouped by destination rank
// (hash_rank of the canonical key). d_keys stays valid until the next partition call on this engine.
void partition_keys_by_rank(Engine& e, const Column& c, int64_t n, int world, uint64_t** d_keys, int64_t* counts,
                            int64_t* n_nulls, int& launches);

// the same partition in two halves for the push shuffle (comm.cpp): counts first, then the scatter straight into the
// destination ranks' receive buffers (one pointer per part, peer memory)
// range_min != nullptr: partition by value range, part = (key - *range_min) / range_span (dense Int64 keys)
void push_partition_hist(Engine& e, const Column& c, int64_t n, int world, int64_t* counts, int64_t* n_nulls, int& launches,
                         const long long* range_min = nullptr, unsigned long long range_span = 1);
void push_partition_scatter(Engine& e, const Column& c, int64_t n, int world, const unsigned long long* first_index, uint64_t* const* d_outs,
                            int& launches, const long long* range_min = nullptr, unsigned long long range_span = 1);
// the exchange of the distributed sort: raw keys (+ payload of 4 / 8 bytes) to the rank whose key range holds them
void split_partition_hist(Engine& e, const uint64_t* d_keys, int64_t n, int world, const uint64_t* d_splitters, int64_t* counts, int& launches);
void split_partition_scatter(Engine& e, const uint64_t* d_keys, const void* d_payload, int pay_bytes, int64_t n, int world,
                             const uint64_t* d_splitters, const unsigned long long* first_index, uint64_t* const* d_key_outs,
                             uint8_t* const* d_pay_outs, int& launches);
bool column_minmax_i64(Engine& e, const Column& c, int64_t n, long long* mn, long long* mx, unsigned long long* n_valid, int& launches);

// hashing.cu: same for Utf8 / composite keys, as 24-byte fingerprint records {h1, h2, has_null}
void partition_fingerprints_by_rank(Engine& e, Table& t, const std::vector<std::string>& names, int world, void** d_records, int64_t* counts,
                                    int& launches);

}  // namespace tg
