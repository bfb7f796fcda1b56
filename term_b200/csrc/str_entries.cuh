// Per-row string entries -> a Utf8 column's Arrow buffers: what the Parquet BYTE_ARRAY path (parquet.cu) and the Arrow
// dictionary / Utf8View paths (tables.cu) share. A producer stages the bytes it decodes from into ONE device block, writes
// one entry {staging offset, length} per row and the byte total of every 1024-row block (its locate kernel); the rest is
// append_utf8_from_entries (parquet.cu).
#pragma once
#include <algorithm>

#include "engine.hpp"

namespace tg {

struct PqBlock {
    uint64_t src_off;     // PLAIN: byte offset in the staging buffer of the block's first non-NULL value (BOOLEAN: bit offset)
    uint32_t first_row;   // chunk-relative
    uint32_t n_rows;      // <= PQ_BLOCK_ROWS
    uint32_t first_dense; // dictionary: dense index (inside the block's section) of the block's first non-NULL value
    uint32_t run_lo, run_hi;  // dictionary: the section's runs [run_lo, run_hi) in the run table; run_hi == 0: a PLAIN block
    uint32_t pad;
};
constexpr int PQ_BLOCK_ROWS = 1024, PQ_THREADS = 256;

// {byte offset in the staging buffer : 40 bits | length : 24 bits}; strings of 16 MiB or more are refused
__host__ __device__ inline uint64_t pq_str_ent(uint64_t off, uint32_t len) { return off | ((uint64_t)len << 40); }
constexpr uint32_t PQ_STR_MAX_LEN = (1u << 24) - 1u;
constexpr uint64_t PQ_STAGE_MAX = (uint64_t)1 << 40;

// staged sections and device tables start 16-byte aligned
inline size_t r16(size_t x) { return (x + 15) & ~(size_t)15; }

// error flags a locate kernel raises (and clamps past); the host turns them into a status
constexpr uint32_t STR_ERR_RANGE = 1u;  // an index / view outside the dictionary / its data buffer: TG_ERR_INVALID_ARG
constexpr uint32_t STR_ERR_LONG = 2u;   // a string of 16 MiB or more: TG_ERR_UNSUPPORTED

// the locate kernels' launch shape: one warp per block, a grid-stride loop over the blocks
inline int pq_str_grid(const Engine& e, int64_t n_blocks) {
    const int64_t w = PQ_THREADS / 32;
    return (int)std::max<int64_t>(1, std::min<int64_t>((n_blocks + w - 1) / w, (int64_t)e.sm_count * 8));
}

// Device tables of one append; all of them live in blocks freed through Engine::deferred_free.
struct Utf8Entries {
    const uint8_t* stage = nullptr;         // the bytes the entries point into
    const PqBlock* blocks = nullptr;        // [n_blocks]
    int64_t n_blocks = 0;
    const uint64_t* row_ent = nullptr;      // [num_values], written by the locate kernel
    unsigned long long* block_bytes = nullptr;  // [n_blocks], written by the locate kernel
    unsigned long long* block_base = nullptr;   // [n_blocks + 1], scratch of the block scan
    const uint32_t* err = nullptr;          // the locate kernel's STR_ERR_* flags; nullptr: it raises none
};

// After the locate kernel (queued on e.copy_stream): pq_block_scan_kernel over the block totals, the byte total (and the
// error flag) read back, the 2 GiB check, the column's value / offset buffers reserved, pq_str_write_kernel, and the
// column's value_bytes / last_offset / n_rows. Validity is the caller's. Returns the error flag: when it is not 0,
// nothing was appended. The caller holds the engine's lock (an AppendTxn).
uint32_t append_utf8_from_entries(Engine& e, Column& c, const Utf8Entries& x, int64_t num_values);

}  // namespace tg
