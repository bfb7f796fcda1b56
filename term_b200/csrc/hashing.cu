// K3 / K5 — GPU hash tables for distinct / unique / primary-key counts, foreign-key anti-joins and grouped
// completeness.
//
// Replaces  COUNT(DISTINCT c), COUNT(DISTINCT (a, b)), GROUP BY .. COUNT(*)     constraints/uniqueness.rs:549-718
//           COUNT(c), COUNT(DISTINCT c)                                          analyzers/basic/distinctness.rs:113
//           LEFT JOIN .. WHERE parent IS NULL -> COUNT(*), COUNT(DISTINCT child)  constraints/foreign_key.rs:165-172
//           GROUP BY g.. COUNT(*), COUNT(c)                                      analyzers/basic/grouped_completeness.rs:131
//
// Keys: a single Int64 / Float64 column is keyed EXACTLY by its 64-bit value (open addressing, linear
// probing, 64-bit atomicCAS). Utf8 and multi-column keys are keyed by a 128-bit fingerprint of the tuple
// (two independent 64-bit hashes; NULL components hash as a tag so NULL is "a value" where SQL makes it
// one). Counting is incremental: the first insert of a key adds one distinct and one singleton, the
// second removes the singleton, so no pass over the table is needed afterwards.
// Round-1 layout: one table in HBM (capacity = next pow2 >= 2n); the radix-partitioned shared-memory
// variant (SURVEY §7.7) is the planned optimisation.
#include <algorithm>
#include <cstring>

#include "engine.hpp"
#include "hash_common.cuh"
#include "hashpart.hpp"

namespace tg {

// ---------------------------------------------------------------- path A: exact 64-bit keys ----
// MASK: also inserts each key that reaches a count of two into the repeated-key table R (key-level row verdicts)
template <bool MASK>
__global__ void __launch_bounds__(HASH_THREADS) insert64_kernel(const uint64_t* values, const uint32_t* validity,
                                                                int64_t n, int is_f64, unsigned long long* keys,
                                                                uint32_t* counts, uint64_t mask, HashCounters* ctr, RepTab R) {
    unsigned long long d = 0, sp = 0, sm = 0, nulls = 0, special = 0;
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x) {
        if (!row_valid(validity, row)) {
            ++nulls;
            continue;
        }
        uint64_t key = values[row];
        if (is_f64) key = canon_f64(key);
        if (key == EMPTY64) {
            ++special;
            continue;
        }
        uint64_t slot = fmix64(key) & mask;
        while (true) {
            const unsigned long long prev = atomicCAS(&keys[slot], EMPTY64, (unsigned long long)key);
            if (prev == EMPTY64 || prev == key) {
                const uint32_t old = atomicAdd(&counts[slot], 1u);
                if (old == 0) {
                    ++d;
                    ++sp;
                } else if (old == 1) {
                    ++sm;
                    if (MASK) rep_insert64(R, key);
                }
                break;
            }
            slot = (slot + 1) & mask;
        }
    }
    flush_counter(d, &ctr->distinct_nonnull);
    flush_counter(sp, &ctr->singles_plus);
    flush_counter(sm, &ctr->singles_minus);
    flush_counter(nulls, &ctr->any_null_rows);
    flush_counter(special, &ctr->special);
}

// ---------------------------------------------------------------- path B: 128-bit fingerprints ----
// fixed-width column -> fingerprint update; nullflag[row] |= 1 when the component is NULL
__global__ void fp_fixed_kernel(const uint8_t* values, const uint32_t* validity, int64_t n, int dtype, int first,
                                Fp* fp, uint8_t* nullflag) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x) {
        Fp acc = first ? Fp{0, 0} : fp[row];
        if (!row_valid(validity, row)) {
            fp_combine(acc, NULL_TAG1, NULL_TAG2, first);
            nullflag[row] = first ? 1 : (nullflag[row] | 1);
        } else {
            uint64_t v;
            switch (dtype) {
                case TG_INT64: v = reinterpret_cast<const uint64_t*>(values)[row]; break;
                case TG_FLOAT64: v = canon_f64(reinterpret_cast<const uint64_t*>(values)[row]); break;
                case TG_INT32: v = (uint64_t)(int64_t)reinterpret_cast<const int32_t*>(values)[row]; break;
                case TG_FLOAT32: v = canon_f64((uint64_t)__double_as_longlong((double)reinterpret_cast<const float*>(values)[row])); break;
                default: v = (reinterpret_cast<const uint32_t*>(values)[row >> 5] >> (row & 31)) & 1u; break;  // TG_BOOL
            }
            fp_combine(acc, v, v ^ 0x5851f42d4c957f2dull, first);
            if (first) nullflag[row] = 0;
        }
        fp[row] = acc;
    }
}

// Utf8 column: two independent multiplicative hashes over the bytes (8 at a time), length-seeded
__global__ void fp_utf8_kernel(const int32_t* offsets, const uint8_t* bytes, const uint32_t* validity, int64_t n, int first,
                               Fp* fp, uint8_t* nullflag) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x) {
        Fp acc = first ? Fp{0, 0} : fp[row];
        if (!row_valid(validity, row)) {
            fp_combine(acc, NULL_TAG1, NULL_TAG2, first);
            nullflag[row] = first ? 1 : (nullflag[row] | 1);
        } else {
            const int32_t b = offsets[row], e = offsets[row + 1];
            uint64_t a = 0x736f6d6570736575ull ^ (uint64_t)(e - b), c = 0x646f72616e646f6dull + (uint64_t)(e - b) * 0x100000001b3ull;
            int32_t p = b;
            for (; p + 8 <= e; p += 8) {
                uint64_t w = 0;
#pragma unroll
                for (int k = 0; k < 8; ++k) w |= (uint64_t)bytes[p + k] << (8 * k);
                a = (a ^ w) * 0x9fb21c651e98df25ull;
                a ^= a >> 29;
                c = (c + w) * 0xc2b2ae3d27d4eb4full;
                c ^= c >> 31;
            }
            uint64_t w = 0;
            for (int k = 0; p + k < e; ++k) w |= (uint64_t)bytes[p + k] << (8 * k);
            a = (a ^ w) * 0x9fb21c651e98df25ull;
            c = (c + w) * 0xc2b2ae3d27d4eb4full;
            fp_combine(acc, fmix64(a), fmix64(c), first);
            if (first) nullflag[row] = 0;
        }
        fp[row] = acc;
    }
}

template <bool MASK>
__global__ void __launch_bounds__(HASH_THREADS) insert128_kernel(const Fp* fp, const uint8_t* nullflag, int64_t n,
                                                                 Table128 t, HashCounters* ctr, RepTab R) {
    unsigned long long da = 0, dn = 0, sp = 0, sm = 0, nulls = 0;
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x) {
        const bool has_null = nullflag[row] != 0;
        nulls += has_null;
        bool created;
        const uint64_t slot = upsert128(t, fp[row], created);
        const uint32_t old = atomicAdd(&t.counts[slot], 1u);
        if (old == 0) {
            ++da;
            dn += !has_null;
            ++sp;
        } else if (old == 1) {
            ++sm;
            if (MASK) rep_insert128(R, fp[row]);
        }
    }
    flush_counter(da, &ctr->distinct_all);
    flush_counter(dn, &ctr->distinct_nonnull);
    flush_counter(sp, &ctr->singles_plus);
    flush_counter(sm, &ctr->singles_minus);
    flush_counter(nulls, &ctr->any_null_rows);
}

// ---------------------------------------------------------------- foreign key ----
// parent set: keys only (64-bit exact or the h1/h2 pair)
__global__ void __launch_bounds__(HASH_THREADS) build_set64_kernel(const uint64_t* values, const uint32_t* validity,
                                                                   int64_t n, int is_f64, unsigned long long* keys,
                                                                   uint64_t mask, unsigned long long* has_special) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x) {
        if (!row_valid(validity, row)) continue;
        uint64_t key = values[row];
        if (is_f64) key = canon_f64(key);
        if (key == EMPTY64) {
            *has_special = 1;
            continue;
        }
        uint64_t slot = fmix64(key) & mask;
        while (true) {
            const unsigned long long prev = atomicCAS(&keys[slot], EMPTY64, (unsigned long long)key);
            if (prev == EMPTY64 || prev == key) break;
            slot = (slot + 1) & mask;
        }
    }
}

__device__ __forceinline__ bool set64_contains(const unsigned long long* keys, uint64_t mask, uint64_t key) {
    uint64_t slot = fmix64(key) & mask;
    while (true) {
        const unsigned long long v = keys[slot];
        if (v == key) return true;
        if (v == EMPTY64) return false;
        slot = (slot + 1) & mask;
    }
}

// pass 1: count violating child rows; pass 2 (collect != 0): also dedupe violators into vkeys/vcounts and record
// up to max_examples row indices of first occurrences
__global__ void __launch_bounds__(HASH_THREADS) fk_probe64_kernel(const uint64_t* child, const uint32_t* validity, int64_t n,
                                                                  int is_f64, const unsigned long long* pkeys, uint64_t pmask,
                                                                  const unsigned long long* parent_has_special, int allow_nulls,
                                                                  int collect, unsigned long long* vkeys, uint32_t* vcounts,
                                                                  uint64_t vmask, int64_t* examples, int max_examples,
                                                                  HashCounters* ctr) {
    unsigned long long viol = 0, nullc = 0, dist = 0;
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x) {
        if (!row_valid(validity, row)) {
            ++nullc;
            if (!allow_nulls) ++viol;
            continue;
        }
        uint64_t key = child[row];
        if (is_f64) key = canon_f64(key);
        const bool found = key == EMPTY64 ? (*parent_has_special != 0) : set64_contains(pkeys, pmask, key);
        if (found) continue;
        ++viol;
        if (collect) {
            if (key == EMPTY64) {
                if (atomicAdd(&ctr->special, 1ull) == 0) {
                    ++dist;
                    const unsigned long long idx = atomicAdd(&ctr->n_examples, 1ull);
                    if (idx < (unsigned long long)max_examples) examples[idx] = row;
                }
                continue;
            }
            uint64_t slot = fmix64(key) & vmask;
            while (true) {
                const unsigned long long prev = atomicCAS(&vkeys[slot], EMPTY64, (unsigned long long)key);
                if (prev == EMPTY64 || prev == key) {
                    if (atomicAdd(&vcounts[slot], 1u) == 0) {
                        ++dist;
                        const unsigned long long idx = atomicAdd(&ctr->n_examples, 1ull);
                        if (idx < (unsigned long long)max_examples) examples[idx] = row;
                    }
                    break;
                }
                slot = (slot + 1) & vmask;
            }
        }
    }
    flush_counter(viol, &ctr->violations);
    flush_counter(nullc, &ctr->null_children);
    if (collect) flush_counter(dist, &ctr->distinct_all);
}

// fingerprint variants (Utf8 keys)
__global__ void __launch_bounds__(HASH_THREADS) build_set128_kernel(const Fp* fp, const uint8_t* nullflag, int64_t n, Table128 t) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x) {
        if (nullflag[row]) continue;
        bool created;
        upsert128(t, fp[row], created);
    }
}
__device__ __forceinline__ bool set128_contains(const Table128& t, Fp f) {
    uint64_t a = f.h1 == EMPTY64 ? 0 : f.h1, b = f.h2 == EMPTY64 ? 0 : f.h2;
    uint64_t slot = (a ^ (b >> 32)) & t.mask;
    while (true) {
        const unsigned long long v = t.h1[slot];
        if (v == EMPTY64) return false;
        if (v == a && t.h2[slot] == b) return true;
        slot = (slot + 1) & t.mask;
    }
}
__global__ void __launch_bounds__(HASH_THREADS) fk_probe128_kernel(const Fp* fp, const uint8_t* nullflag, int64_t n, Table128 parent,
                                                                   int allow_nulls, int collect, Table128 viol_t, int64_t* examples,
                                                                   int max_examples, HashCounters* ctr) {
    unsigned long long viol = 0, nullc = 0, dist = 0;
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x) {
        if (nullflag[row]) {
            ++nullc;
            if (!allow_nulls) ++viol;
            continue;
        }
        if (set128_contains(parent, fp[row])) continue;
        ++viol;
        if (collect) {
            bool created;
            const uint64_t slot = upsert128(viol_t, fp[row], created);
            if (atomicAdd(&viol_t.counts[slot], 1u) == 0) {
                ++dist;
                const unsigned long long idx = atomicAdd(&ctr->n_examples, 1ull);
                if (idx < (unsigned long long)max_examples) examples[idx] = row;
            }
        }
    }
    flush_counter(viol, &ctr->violations);
    flush_counter(nullc, &ctr->null_children);
    if (collect) flush_counter(dist, &ctr->distinct_all);
}

// ---------------------------------------------------------------- key-level row verdicts ----
// The key of a row: the canonical 64-bit value or the fingerprint (FP; nullflag given for a single-column key, whose NULL
// rows have no key; a composite key is a value in every row). validity: the single key column's (nullptr: every row valid).
struct RowKeys {
    const uint64_t* values;
    const uint32_t* validity;
    int is_f64;
    const Fp* fp;
    const uint8_t* nullflag;
};
template <bool FP>
__device__ __forceinline__ bool row_key_valid(const RowKeys& k, int64_t row) {
    return FP ? !(k.nullflag && k.nullflag[row]) : row_valid(k.validity, row);
}
template <bool FP>
__device__ __forceinline__ unsigned long long* row_rep_cell(const RepTab& R, const RowKeys& k, int64_t row) {
    if (!R.h1) return nullptr;  // no repeated key: the key is not read
    if (FP) return rep_cell128(R, k.fp[row]);
    const uint64_t v = k.values[row];
    return rep_cell64(R, k.is_f64 ? canon_f64(v) : v);
}

__global__ void rep_mark_kernel(RepTab R, uint64_t key) { rep_insert64(R, key); }

// row pass 1: the lowest row of every repeated key
template <bool FP>
__global__ void __launch_bounds__(HASH_THREADS) rep_min_rows_kernel(RowKeys k, int64_t n, RepTab R) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x) {
        if (!row_key_valid<FP>(k, row)) continue;
        unsigned long long* cell = row_rep_cell<FP>(R, k, row);
        if (cell) atomicMin(cell, (unsigned long long)row);
    }
}
// row pass 2: one warp per 32-row word; DUPLICATE = the key is in R, FIRST = it is not, or this row is its lowest
template <bool FP>
__global__ void __launch_bounds__(HASH_THREADS) rep_verdict_kernel(RowKeys k, int64_t n, RepTab R, VerdictOut dup, VerdictOut first) {
    const int64_t n_words = (n + 31) >> 5, warps = (int64_t)gridDim.x * (HASH_THREADS / 32);
    if (!R.h1) {  // no repeated key: DUPLICATE = 0 and FIRST = validity, one thread per word, no key read
        for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (int64_t)gridDim.x * blockDim.x) {
            const int64_t rem = n - 32 * w;
            const uint32_t v = (k.validity ? k.validity[w] : 0xffffffffu) & (rem >= 32 ? 0xffffffffu : (1u << rem) - 1u);
            if (dup.values) dup.values[w] = 0u;
            if (dup.validity) dup.validity[w] = v;
            if (first.values) first.values[w] = v;
            if (first.validity) first.validity[w] = v;
        }
        return;
    }
    for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_words; w += warps) {
        const int64_t row = 32 * w + (threadIdx.x & 31);
        const bool valid = row < n && row_key_valid<FP>(k, row);
        const unsigned long long* cell = valid ? row_rep_cell<FP>(R, k, row) : nullptr;
        store_verdict_word(w, cell != nullptr, valid, dup);
        store_verdict_word(w, !cell || *cell == (unsigned long long)row, valid, first);
    }
}

// FK: bit = the child row's key is in the exact table of distinct orphan keys that the probe path built
struct Key64 {
    const uint64_t* values;
    int is_f64;
    const unsigned long long* vkeys;  // nullptr: no key violates
    uint64_t vmask;
    int shift;           // slot = (fmix64(key) >> shift) & vmask, as the path's probe kernel placed it
    int special_orphan;  // the EMPTY-sentinel key (Int64 -1), kept out of the table, has no parent
    __device__ __forceinline__ bool orphan(int64_t row) const {
        uint64_t key = values[row];
        if (is_f64) key = canon_f64(key);
        if (key == EMPTY64) return special_orphan != 0;
        if (!vkeys) return false;
        uint64_t slot = (fmix64(key) >> shift) & vmask;
        for (uint64_t probes = 0; probes <= vmask; ++probes) {
            const unsigned long long v = vkeys[slot];
            if (v == key) return true;
            if (v == EMPTY64) return false;
            slot = (slot + 1) & vmask;
        }
        return false;
    }
};
struct Fp128 {
    const Fp* fp;
    Table128 vtab;  // h1 == nullptr: no key violates
    __device__ __forceinline__ bool orphan(int64_t row) const { return vtab.h1 && set128_contains(vtab, fp[row]); }
};
template <class K>
__global__ void __launch_bounds__(HASH_THREADS) fk_orphan_rows_kernel(K k, const uint32_t* validity, int64_t n, VerdictOut out) {
    const int64_t n_words = (n + 31) >> 5, warps = (int64_t)gridDim.x * (HASH_THREADS / 32);
    for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_words; w += warps) {
        const int64_t row = 32 * w + (threadIdx.x & 31);
        const bool valid = row < n && row_valid(validity, row);
        store_verdict_word(w, valid && k.orphan(row), valid, out);
    }
}

// ================================================================== host side ==================
static uint64_t pow2_at_least(uint64_t x) {
    uint64_t p = 1024;
    while (p < x) p <<= 1;
    return p;
}
static size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static int grid_for(Engine& e, int64_t n) {
    const int64_t blocks = (n + HASH_THREADS - 1) / HASH_THREADS;
    return (int)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)e.sm_count * 8));
}

struct Timer {
    Engine& e;
    Plan& p;
    Timer(Engine& e_, Plan& p_) : e(e_), p(p_) { cudaEventRecord(e.ev[4], e.stream); }
    void stop(int launches) {
        cudaEventRecord(e.ev[5], e.stream);
        cudaStreamSynchronize(e.stream);
        float ms = 0;
        cudaEventElapsedTime(&ms, e.ev[4], e.ev[5]);
        p.stats.hash_ms += ms;
        p.stats.gpu_ms += ms;
        p.stats.launches += launches;
        e.launches += launches;
    }
};

static Column* need_col(Table& t, const std::string& name) {
    Column* c = t.find(name);
    if (!c) throw Error(TG_ERR_COLUMN_NOT_FOUND, "Schema error: No field named " + name + ". Valid fields are " + t.valid_fields() + ".");
    return c;
}

static uint64_t col_bytes(const Column& c, int64_t n) {
    uint64_t b = c.validity.p ? (uint64_t)(n + 7) / 8 : 0;
    if (c.dtype == TG_UTF8) return b + (uint64_t)(n + 1) * 4 + (uint64_t)c.value_bytes;
    if (c.dtype == TG_BOOL) return b + (uint64_t)(n + 7) / 8;
    return b + (uint64_t)n * c.elem_bytes();
}

// fingerprints of a tuple of columns into scratch; returns launches
static int compute_fingerprints(Engine& e, Table& t, const std::vector<Column*>& cols, Fp* d_fp, uint8_t* d_null) {
    const int64_t n = t.n_rows;
    const int grid = grid_for(e, n);
    int launches = 0;
    for (size_t i = 0; i < cols.size(); ++i) {
        Column* c = cols[i];
        if (c->dtype == TG_UTF8)
            fp_utf8_kernel<<<grid, HASH_THREADS, 0, e.stream>>>((const int32_t*)c->offsets.p, c->values.p,
                                                                (const uint32_t*)c->validity.p, n, i == 0, d_fp, d_null);
        else
            fp_fixed_kernel<<<grid, HASH_THREADS, 0, e.stream>>>(c->values.p, (const uint32_t*)c->validity.p, n, c->dtype,
                                                                 i == 0, d_fp, d_null);
        TG_CUDA(cudaGetLastError());
        ++launches;
    }
    return launches;
}

// ---------------------------------------------------------------- fingerprint shuffle (multi-GPU, Utf8 / composite keys) ----
struct FpRecord {
    unsigned long long h1, h2, has_null;
};
constexpr int FPS_THREADS = 256, FPS_ROWS = 4, FPS_MAX_PARTS = 1024;

__global__ void __launch_bounds__(FPS_THREADS) fp_rank_hist_kernel(const Fp* fp, int64_t n, uint32_t parts, unsigned long long* hist) {
    __shared__ uint32_t s_hist[FPS_MAX_PARTS];
    for (int i = threadIdx.x; i < (int)parts; i += FPS_THREADS) s_hist[i] = 0;
    __syncthreads();
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x)
        atomicAdd(&s_hist[hash_rank(fp[row].h1, parts)], 1u);
    __syncthreads();
    for (int i = threadIdx.x; i < (int)parts; i += FPS_THREADS)
        if (s_hist[i]) atomicAdd(&hist[i], (unsigned long long)s_hist[i]);
}
__global__ void fp_prefix_kernel(const unsigned long long* hist, uint32_t parts, unsigned long long* offsets, unsigned long long* cursors) {
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (uint32_t i = 0; i < parts; ++i) {
            offsets[i] = run;
            cursors[i] = run;
            run += hist[i];
        }
        offsets[parts] = run;
    }
}
__global__ void __launch_bounds__(FPS_THREADS) fp_rank_scatter_kernel(const Fp* fp, const uint8_t* nullflag, int64_t n, uint32_t parts,
                                                                      unsigned long long* cursors, FpRecord* out) {
    __shared__ uint32_t s_cnt[FPS_MAX_PARTS];
    __shared__ unsigned long long s_base[FPS_MAX_PARTS];
    const int64_t tile_rows = (int64_t)FPS_THREADS * FPS_ROWS;
    for (int64_t base = (int64_t)blockIdx.x * tile_rows; base < n; base += (int64_t)gridDim.x * tile_rows) {
        for (int i = threadIdx.x; i < (int)parts; i += FPS_THREADS) s_cnt[i] = 0;
        __syncthreads();
        uint32_t part[FPS_ROWS], rank[FPS_ROWS];
#pragma unroll
        for (int k = 0; k < FPS_ROWS; ++k) {
            const int64_t row = base + (int64_t)k * FPS_THREADS + threadIdx.x;
            part[k] = 0xffffffffu;
            if (row < n) {
                part[k] = hash_rank(fp[row].h1, parts);
                rank[k] = atomicAdd(&s_cnt[part[k]], 1u);
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < (int)parts; i += FPS_THREADS)
            if (s_cnt[i]) s_base[i] = atomicAdd(&cursors[i], (unsigned long long)s_cnt[i]);
        __syncthreads();
#pragma unroll
        for (int k = 0; k < FPS_ROWS; ++k) {
            const int64_t row = base + (int64_t)k * FPS_THREADS + threadIdx.x;
            if (part[k] != 0xffffffffu) out[s_base[part[k]] + rank[k]] = FpRecord{fp[row].h1, fp[row].h2, nullflag[row] ? 1ull : 0ull};
        }
        __syncthreads();
    }
}
__global__ void fp_unpack_kernel(const FpRecord* rec, int64_t n, Fp* fp, uint8_t* nullflag) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x) {
        fp[row] = Fp{rec[row].h1, rec[row].h2};
        nullflag[row] = rec[row].has_null ? 1 : 0;
    }
}

// tg_table_partition_fingerprints: records grouped by destination rank in the engine's shuffle buffer
void partition_fingerprints_by_rank(Engine& e, Table& t, const std::vector<std::string>& names, int world, void** d_records, int64_t* counts,
                                    int& launches) {
    if (world < 1 || world > FPS_MAX_PARTS) throw Error(TG_ERR_INVALID_ARG, "world size must be in 1..1024");
    std::vector<Column*> cols;
    for (auto& nm : names) cols.push_back(need_col(t, nm));
    if (cols.empty()) throw Error(TG_ERR_INVALID_ARG, "no key columns");
    const int64_t n = t.n_rows;
    const size_t rec_b = round_up((size_t)std::max<int64_t>(n, 1) * sizeof(FpRecord), 256), meta_b = round_up((size_t)(3 * (FPS_MAX_PARTS + 1)) * 8, 256);
    const size_t need = rec_b + meta_b;
    if (need > e.shuffle_cap) {
        TG_CUDA(cudaStreamSynchronize(e.stream));
        if (e.d_shuffle) TG_CUDA(cudaFree(e.d_shuffle));
        e.d_shuffle = nullptr;
        e.shuffle_cap = 0;
        TG_CUDA(cudaMalloc(&e.d_shuffle, need));
        e.shuffle_cap = need;
    }
    unsigned long long* hist = (unsigned long long*)(e.d_shuffle + rec_b);
    unsigned long long* offsets = hist + (FPS_MAX_PARTS + 1);
    unsigned long long* cursors = offsets + (FPS_MAX_PARTS + 1);
    TG_CUDA(cudaMemsetAsync(hist, 0, meta_b, e.stream));
    if (n > 0) {
        const size_t fp_b = round_up((size_t)n * 16, 256), nf_b = round_up((size_t)n, 256);
        uint8_t* scr = e.scratch(fp_b + nf_b);
        Fp* d_fp = (Fp*)scr;
        uint8_t* d_null = scr + fp_b;
        launches += compute_fingerprints(e, t, cols, d_fp, d_null);
        fp_rank_hist_kernel<<<grid_for(e, n), FPS_THREADS, 0, e.stream>>>(d_fp, n, (uint32_t)world, hist);
        fp_prefix_kernel<<<1, 32, 0, e.stream>>>(hist, (uint32_t)world, offsets, cursors);
        const int64_t tiles = (n + FPS_THREADS * FPS_ROWS - 1) / (FPS_THREADS * FPS_ROWS);
        fp_rank_scatter_kernel<<<(int)std::max<int64_t>(1, std::min<int64_t>(tiles, (int64_t)e.sm_count * 8)), FPS_THREADS, 0, e.stream>>>(
            d_fp, d_null, n, (uint32_t)world, cursors, (FpRecord*)e.d_shuffle);
        TG_CUDA(cudaGetLastError());
        launches += 3;
    }
    std::vector<unsigned long long> h((size_t)world);
    TG_CUDA(cudaMemcpyAsync(h.data(), hist, h.size() * 8, cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    for (int i = 0; i < world; ++i) counts[i] = (int64_t)h[i];
    *d_records = e.d_shuffle;
}

// ---------------------------------------------------------------- key-level row verdicts (host) ----
static int word_grid(Engine& e, int64_t n) {
    const int64_t blocks = ((n + 31) / 32 + HASH_THREADS / 32 - 1) / (HASH_THREADS / 32);
    return (int)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)e.sm_count * 8));
}

// R in one recycled device block: h1 [cap], h2 [cap] (fingerprints only), minrow [cap], empty_key [2], fill [1]
static size_t rep_bytes(uint64_t cap, bool fp) { return (size_t)cap * 8 * (fp ? 3 : 2) + 24; }
void rep_reset(Engine& e, const RepTab& R) {
    TG_CUDA(cudaMemsetAsync(R.h1, 0xFF, rep_bytes(R.mask + 1, R.h2 != nullptr), e.stream));
    TG_CUDA(cudaMemsetAsync(R.empty_key, 0, 8, e.stream));
    TG_CUDA(cudaMemsetAsync(R.fill, 0, 8, e.stream));
}
void rep_mark(Engine& e, const RepTab& R, uint64_t key) {
    rep_mark_kernel<<<1, 1, 0, e.stream>>>(R, key);
    TG_CUDA(cudaGetLastError());
}
struct RepBuf {
    Engine& e;
    RepTab R;
    uint8_t* block = nullptr;
    size_t bytes = 0;
    explicit RepBuf(Engine& e_) : e(e_) {}
    ~RepBuf() { release(); }
    void release() {
        if (block) e.dev_free(block, bytes);
        block = nullptr;
    }
    void alloc(uint64_t cap, bool fp) {
        release();
        bytes = rep_bytes(cap, fp);
        block = e.dev_alloc(bytes);
        unsigned long long* q = reinterpret_cast<unsigned long long*>(block);
        R.h1 = q;
        R.h2 = fp ? q + cap : nullptr;
        R.minrow = q + cap * (fp ? 2 : 1);
        R.empty_key = q + cap * (fp ? 3 : 2);
        R.fill = R.empty_key + 2;
        R.mask = cap - 1;
    }
};
constexpr uint64_t REP_CAP0 = 1u << 20;

static VerdictOut verdict_out(const std::shared_ptr<RowMask>& m) {
    VerdictOut o;
    if (m) {
        o.values = reinterpret_cast<uint32_t*>(m->values);
        o.validity = reinterpret_cast<uint32_t*>(m->validity);
    }
    return o;
}

// the job's repeated-key count after the counting pass: the keys R has to hold
static uint64_t count_distinct(Engine& e, Table& t, Plan& p, Agg& a, const std::vector<Column*>& cols, Column* shard, const RepTab* R,
                               Fp*& d_fp, uint8_t*& d_null) {
    const int64_t n = t.n_rows;
    const bool from_records = shard != nullptr;
    const bool exact64 = cols.size() == 1 && (cols[0]->dtype == TG_INT64 || cols[0]->dtype == TG_FLOAT64);
    if (exact64 && n > (1 << 20)) {
        // large key column: dense Int64 ranges are counted in bitmaps (hashpart.cu); anything else is hashed, radix-sorted by
        // its low hash bits and de-duplicated in shared memory (hashsort.cu) — or, for hot keys, radix-partitioned and
        // de-duplicated bucket by bucket in an L2-resident table (hashpart.cu)
        Distinct64Result r;
        Timer tm(e, p);
        int launches = 0;
        bool ok = distinct64_dense(e, *cols[0], n, (a.flags & 1) != 0, r, launches, R);
        if (!ok && (size_t)n > distinct64_min_rows()) ok = distinct64_sorted(e, *cols[0], n, r, launches, R);
        if (!ok && (size_t)n > distinct64_min_rows()) ok = distinct64_partitioned(e, *cols[0], n, r, launches, R);
        tm.stop(launches);
        if (ok) {
            const uint64_t singles = r.distinct - r.dup_keys;
            a.u[1] = r.distinct;
            a.u[2] = singles + (r.nulls == 1 ? 1 : 0);  // the NULL group of GROUP BY
            a.u[3] = r.nulls;
            a.u[4] = r.nulls;
            a.u[5] = r.distinct + (r.nulls > 0 ? 1 : 0);
            return r.dup_keys;
        }
        // a bucket table overflowed (adversarial hash skew): fall through to the single-table path
    }
    const uint64_t cap = pow2_at_least((uint64_t)n * 2);
    HashCounters h{};
    Timer tm(e, p);
    int launches = 0;
    if (R) rep_reset(e, *R);
    if (exact64) {
        const size_t keys_b = cap * 8, cnt_b = cap * 4;
        uint8_t* scr = e.scratch(keys_b + cnt_b + 256);
        unsigned long long* keys = (unsigned long long*)scr;
        uint32_t* counts = (uint32_t*)(scr + keys_b);
        HashCounters* d_ctr = (HashCounters*)(scr + keys_b + cnt_b);
        TG_CUDA(cudaMemsetAsync(keys, 0xFF, keys_b, e.stream));
        TG_CUDA(cudaMemsetAsync(counts, 0, cnt_b + 256, e.stream));
        const uint64_t* vals = (const uint64_t*)cols[0]->values.p;
        const uint32_t* valid = (const uint32_t*)cols[0]->validity.p;
        const int is_f64 = cols[0]->dtype == TG_FLOAT64;
        if (R)
            insert64_kernel<true><<<grid_for(e, n), HASH_THREADS, 0, e.stream>>>(vals, valid, n, is_f64, keys, counts, cap - 1, d_ctr, *R);
        else
            insert64_kernel<false><<<grid_for(e, n), HASH_THREADS, 0, e.stream>>>(vals, valid, n, is_f64, keys, counts, cap - 1, d_ctr, RepTab{});
        TG_CUDA(cudaGetLastError());
        launches = 1;
        TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
        tm.stop(launches);
        uint64_t distinct_nonnull = h.distinct_nonnull, singles = h.singles_plus - h.singles_minus;
        if (h.special) {
            distinct_nonnull += 1;
            singles += h.special == 1;
        }
        // the Int64 value -1 is the table's EMPTY word: counted apart, and marked repeated by hand
        if (R && h.special > 1) rep_mark(e, *R, EMPTY64);
        const uint64_t nulls = h.any_null_rows;
        a.u[1] = distinct_nonnull;
        a.u[2] = singles + (nulls == 1 ? 1 : 0);  // the NULL group of GROUP BY
        a.u[3] = nulls;
        a.u[4] = nulls;
        a.u[5] = distinct_nonnull + (nulls > 0 ? 1 : 0);
        return h.singles_minus + (h.special > 1 ? 1 : 0);
    }
    const size_t fp_b = round_up((size_t)n * 16, 256), nf_b = round_up((size_t)n, 256);
    const size_t h_b = cap * 8, cnt_b = cap * 4;
    uint8_t* scr = e.scratch(fp_b + nf_b + 2 * h_b + cnt_b + 256);
    d_fp = (Fp*)scr;
    d_null = scr + fp_b;
    Table128 tb{(unsigned long long*)(scr + fp_b + nf_b), (unsigned long long*)(scr + fp_b + nf_b + h_b),
                (uint32_t*)(scr + fp_b + nf_b + 2 * h_b), cap - 1};
    HashCounters* d_ctr = (HashCounters*)(scr + fp_b + nf_b + 2 * h_b + cnt_b);
    TG_CUDA(cudaMemsetAsync(tb.h1, 0xFF, 2 * h_b, e.stream));
    TG_CUDA(cudaMemsetAsync(tb.counts, 0, cnt_b + 256, e.stream));
    if (from_records) {
        fp_unpack_kernel<<<grid_for(e, n), HASH_THREADS, 0, e.stream>>>((const FpRecord*)shard->values.p, n, d_fp, d_null);
        ++launches;
    } else {
        launches += compute_fingerprints(e, t, cols, d_fp, d_null);
    }
    if (R) insert128_kernel<true><<<grid_for(e, n), HASH_THREADS, 0, e.stream>>>(d_fp, d_null, n, tb, d_ctr, *R);
    else insert128_kernel<false><<<grid_for(e, n), HASH_THREADS, 0, e.stream>>>(d_fp, d_null, n, tb, d_ctr, RepTab{});
    TG_CUDA(cudaGetLastError());
    ++launches;
    TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
    tm.stop(launches);
    a.u[1] = h.distinct_nonnull;
    a.u[2] = h.singles_plus - h.singles_minus;
    a.u[3] = h.any_null_rows;
    a.u[4] = h.any_null_rows;
    a.u[5] = h.distinct_all;
    return h.singles_minus;
}

void exec_distinct_job(Engine& e, Table& t, Plan& p, int agg_id) {
    Agg& a = p.aggs[agg_id];
    std::vector<Column*> cols;
    // a hash-shuffled shard of a Utf8 / composite key arrives as ONE column of fingerprint records
    Column* shard = t.find("tg_fp");
    const bool from_records = shard && shard->dtype == TG_FP128;
    if (from_records) cols.push_back(shard);
    else
        for (auto& name : a.cols) cols.push_back(need_col(t, name));
    if (!from_records) shard = nullptr;
    const int64_t n = t.n_rows;
    a.u[0] = (uint64_t)n;
    for (auto* c : cols) p.stats.bytes_scanned += from_records ? (uint64_t)n * sizeof(FpRecord) : col_bytes(*c, n);
    // key-level row verdicts of the rows of this table (a shard of keys shuffled here from other ranks has none: the
    // export reports it); a NULL single-column key has none either, a composite key is a value in every row
    const bool verdicts = (a.key_rows & ((1 << TG_KEY_ROWS_DUPLICATE) | (1 << TG_KEY_ROWS_FIRST))) && a.redirect[0].empty() && !from_records;
    const bool single = cols.size() == 1;
    const bool emit_validity = single && cols[0]->validity.p && cols[0]->null_count > 0;
    if (verdicts)
        for (int k : {TG_KEY_ROWS_DUPLICATE, TG_KEY_ROWS_FIRST})
            if (a.key_rows & (1 << k)) a.key_mask[k] = new_row_mask(e, n, emit_validity);
    if (n == 0) return;
    const bool fp = !(single && (cols[0]->dtype == TG_INT64 || cols[0]->dtype == TG_FLOAT64));
    RepBuf rb(e);
    if (verdicts) rb.alloc(REP_CAP0, fp);
    Fp* d_fp = nullptr;
    uint8_t* d_null = nullptr;
    uint64_t reps = count_distinct(e, t, p, a, cols, shard, verdicts ? &rb.R : nullptr, d_fp, d_null);
    if (!verdicts) return;
    if (reps > REP_CAP0 / 2) {
        // more repeated keys than R holds at load 1/2: repeat the job once with R sized from the now-known count
        rb.alloc(pow2_at_least(reps * 2), fp);
        reps = count_distinct(e, t, p, a, cols, shard, &rb.R, d_fp, d_null);
    }
    // no repeated key (a passing is_unique): no row pass against R, every valid row is the first of its key
    const RepTab R = reps ? rb.R : RepTab{};
    const RowKeys k{fp ? nullptr : (const uint64_t*)cols[0]->values.p, single ? (const uint32_t*)cols[0]->validity.p : nullptr,
                    !fp && cols[0]->dtype == TG_FLOAT64, d_fp, fp && single ? d_null : nullptr};
    const VerdictOut dup = verdict_out(a.key_mask[TG_KEY_ROWS_DUPLICATE]), first = verdict_out(a.key_mask[TG_KEY_ROWS_FIRST]);
    Timer tm(e, p);
    int launches = 1;
    if (reps) {
        if (fp) rep_min_rows_kernel<true><<<grid_for(e, n), HASH_THREADS, 0, e.stream>>>(k, n, R);
        else rep_min_rows_kernel<false><<<grid_for(e, n), HASH_THREADS, 0, e.stream>>>(k, n, R);
        ++launches;
    }
    if (fp) rep_verdict_kernel<true><<<word_grid(e, n), HASH_THREADS, 0, e.stream>>>(k, n, R, dup, first);
    else rep_verdict_kernel<false><<<word_grid(e, n), HASH_THREADS, 0, e.stream>>>(k, n, R, dup, first);
    TG_CUDA(cudaGetLastError());
    tm.stop(launches);
    const int64_t nulls = emit_validity ? (int64_t)a.u[3] : 0;
    for (auto& m : a.key_mask)
        if (m) m->null_count = nulls;
}

// FK orphan rows of a 64-bit child key column (the paths of hashpart.cu call this with their orphan table)
void fk_orphan_rows64(Engine& e, const Column& child, int64_t nc, const unsigned long long* vkeys, uint64_t vmask, int shift,
                      bool special_orphan, const VerdictOut& out, int& launches) {
    if (nc == 0) return;
    const Key64 k{(const uint64_t*)child.values.p, child.dtype == TG_FLOAT64, vkeys, vmask, shift, special_orphan ? 1 : 0};
    fk_orphan_rows_kernel<Key64><<<word_grid(e, nc), HASH_THREADS, 0, e.stream>>>(k, (const uint32_t*)child.validity.p, nc, out);
    TG_CUDA(cudaGetLastError());
    ++launches;
}

// value of a row as the reference prints violation examples (foreign_key.rs:250-290)
static std::string row_to_string(Engine& e, Column& c, int64_t row) {
    if (c.dtype == TG_UTF8) {
        int32_t off[2];
        TG_CUDA(cudaMemcpy(off, c.offsets.p + (size_t)row * 4, 8, cudaMemcpyDeviceToHost));
        std::string s((size_t)(off[1] - off[0]), '\0');
        if (!s.empty()) TG_CUDA(cudaMemcpy(&s[0], c.values.p + off[0], s.size(), cudaMemcpyDeviceToHost));
        return s;
    }
    if (c.dtype == TG_INT64) {
        int64_t v;
        TG_CUDA(cudaMemcpy(&v, c.values.p + (size_t)row * 8, 8, cudaMemcpyDeviceToHost));
        return fmt_i64(v);
    }
    if (c.dtype == TG_FLOAT64) {
        double v;
        TG_CUDA(cudaMemcpy(&v, c.values.p + (size_t)row * 8, 8, cudaMemcpyDeviceToHost));
        return fmt_f64(v);
    }
    if (c.dtype == TG_INT32) {
        int32_t v;
        TG_CUDA(cudaMemcpy(&v, c.values.p + (size_t)row * 4, 4, cudaMemcpyDeviceToHost));
        return fmt_i64(v);
    }
    return "";
}

void exec_fk_job(Engine& e, Plan& p, int agg_id) {
    Agg& a = p.aggs[agg_id];
    auto find_table = [&](const std::string& name) -> Table& {
        auto it = e.tables.find(name);
        if (it == e.tables.end())
            throw Error(TG_ERR_TABLE_NOT_FOUND, "Constraint evaluation failed for 'foreign_key': Foreign key validation query failed: "
                                                "Error during planning: table 'datafusion.public." + name + "' not found");
        return *it->second;
    };
    Table& ct = find_table(a.redirect[0].empty() ? a.cols[0] : a.redirect[0]);
    Table& pt = find_table(a.redirect[1].empty() ? a.cols[2] : a.redirect[1]);
    // hash-shuffled shards of Utf8 key columns (multi-GPU) arrive as ONE column of fingerprint records on both sides
    Column* cshard = a.redirect[0].empty() ? nullptr : ct.find("tg_fp");
    Column* pshard = a.redirect[1].empty() ? nullptr : pt.find("tg_fp");
    const bool from_records = cshard && pshard && cshard->dtype == TG_FP128 && pshard->dtype == TG_FP128;
    Column* cc = from_records ? cshard : need_col(ct, a.cols[1]);
    Column* pc = from_records ? pshard : need_col(pt, a.cols[3]);
    if (cc->dtype != pc->dtype)
        throw Error(TG_ERR_TYPE_MISMATCH, "foreign key columns have different types");
    const int64_t nc = ct.n_rows, np = pt.n_rows;
    p.stats.bytes_scanned += from_records ? (uint64_t)(nc + np) * sizeof(FpRecord) : col_bytes(*cc, nc) + col_bytes(*pc, np);
    const int allow_nulls = a.flags, max_examples = std::max(0, a.iparam);
    // orphan row verdicts cover the child table's rows; keys shuffled here from other ranks are not that table's rows
    VerdictOut orphan;
    const VerdictOut* orphan_rows = nullptr;
    if ((a.key_rows & (1 << TG_KEY_ROWS_ORPHAN)) && a.redirect[0].empty() && a.redirect[1].empty()) {
        const bool emit_validity = cc->validity.p && cc->null_count > 0;
        auto& m = a.key_mask[TG_KEY_ROWS_ORPHAN];
        m = new_row_mask(e, nc, emit_validity);
        m->null_count = emit_validity ? cc->null_count : 0;
        orphan = verdict_out(m);
        orphan_rows = &orphan;
    }
    if (nc == 0) return;
    const bool exact64 = cc->dtype == TG_INT64 || cc->dtype == TG_FLOAT64;
    const uint64_t pcap = pow2_at_least((uint64_t)std::max<int64_t>(np, 1) * 2);
    HashCounters h{};
    Timer tm(e, p);
    int launches = 0;
    std::vector<int64_t> ex_rows;
    if (exact64 && (nc > (1 << 20) || (size_t)np > distinct64_min_rows())) {
        // hashpart.cu: a dense Int64 parent range becomes a bitmap; a parent key set too large for an L2-resident
        // table is radix-partitioned together with the child keys by the same hash bits
        Fk64Result r;
        bool ok = fk64_dense(e, *cc, nc, *pc, np, allow_nulls, max_examples, r, launches, orphan_rows);
        if (!ok && (size_t)np > distinct64_min_rows())
            ok = fk64_partitioned(e, *cc, nc, *pc, np, allow_nulls, max_examples, r, launches, orphan_rows);
        if (ok) {
            tm.stop(launches);
            a.u[0] = r.violations;
            a.u[1] = r.distinct_violations;
            a.u[2] = r.null_children;
            std::vector<std::string> ex;
            if (cc->dtype == TG_INT64) {
                std::vector<int64_t> ks;
                for (uint64_t k : r.example_keys) ks.push_back((int64_t)k);
                std::sort(ks.begin(), ks.end());
                for (int64_t k : ks) ex.push_back(fmt_i64(k));
            } else {
                std::vector<double> ks;
                for (uint64_t k : r.example_keys) {
                    double d;
                    memcpy(&d, &k, 8);
                    ks.push_back(d);
                }
                std::sort(ks.begin(), ks.end(), [](double x, double y) { return x < y || (y != y && x == x); });
                for (double d : ks) ex.push_back(fmt_f64(d));
            }
            uint64_t cnt = ex.size();
            a.blob.resize(8);
            memcpy(a.blob.data(), &cnt, 8);
            for (auto& s : ex) {
                uint32_t L = (uint32_t)s.size();
                size_t o = a.blob.size();
                a.blob.resize(o + 4 + L);
                memcpy(a.blob.data() + o, &L, 4);
                memcpy(a.blob.data() + o + 4, s.data(), L);
            }
            return;
        }
        launches = 0;  // overflow: redo on the single-table path below
    }
    if (exact64) {
        const size_t pk_b = pcap * 8;
        uint8_t* scr = e.scratch(pk_b + 512);
        unsigned long long* pkeys = (unsigned long long*)scr;
        HashCounters* d_ctr = (HashCounters*)(scr + pk_b);
        unsigned long long* d_special = (unsigned long long*)(scr + pk_b + 256);
        TG_CUDA(cudaMemsetAsync(pkeys, 0xFF, pk_b, e.stream));
        TG_CUDA(cudaMemsetAsync(d_ctr, 0, 512, e.stream));
        if (np > 0) {
            build_set64_kernel<<<grid_for(e, np), HASH_THREADS, 0, e.stream>>>((const uint64_t*)pc->values.p, (const uint32_t*)pc->validity.p,
                                                                               np, pc->dtype == TG_FLOAT64, pkeys, pcap - 1, d_special);
            ++launches;
        }
        fk_probe64_kernel<<<grid_for(e, nc), HASH_THREADS, 0, e.stream>>>((const uint64_t*)cc->values.p, (const uint32_t*)cc->validity.p, nc,
                                                                          cc->dtype == TG_FLOAT64, pkeys, pcap - 1, d_special, allow_nulls, 0,
                                                                          nullptr, nullptr, 0, nullptr, 0, d_ctr);
        TG_CUDA(cudaGetLastError());
        ++launches;
        TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
        TG_CUDA(cudaStreamSynchronize(e.stream));
        const uint64_t viol = h.violations;
        const uint64_t key_viol = viol - (allow_nulls ? 0 : h.null_children);
        if (key_viol > 0) {
            // second pass: dedupe the violating keys (table sized from the known count)
            const uint64_t vcap = pow2_at_least(key_viol * 2);
            const size_t vk_b = vcap * 8, vc_b = vcap * 4, ex_b = round_up((size_t)std::max(max_examples, 1) * 8, 256);
            // scratch may move: re-derive every pointer after growing
            scr = e.scratch(pk_b + 512 + vk_b + vc_b + ex_b);
            pkeys = (unsigned long long*)scr;
            d_ctr = (HashCounters*)(scr + pk_b);
            d_special = (unsigned long long*)(scr + pk_b + 256);
            unsigned long long* vkeys = (unsigned long long*)(scr + pk_b + 512);
            uint32_t* vcounts = (uint32_t*)(scr + pk_b + 512 + vk_b);
            int64_t* d_ex = (int64_t*)(scr + pk_b + 512 + vk_b + vc_b);
            TG_CUDA(cudaMemsetAsync(pkeys, 0xFF, pk_b, e.stream));
            TG_CUDA(cudaMemsetAsync(d_ctr, 0, 512, e.stream));
            TG_CUDA(cudaMemsetAsync(vkeys, 0xFF, vk_b, e.stream));
            TG_CUDA(cudaMemsetAsync(vcounts, 0, vc_b + ex_b, e.stream));
            if (np > 0) {
                build_set64_kernel<<<grid_for(e, np), HASH_THREADS, 0, e.stream>>>((const uint64_t*)pc->values.p, (const uint32_t*)pc->validity.p,
                                                                                   np, pc->dtype == TG_FLOAT64, pkeys, pcap - 1, d_special);
                ++launches;
            }
            fk_probe64_kernel<<<grid_for(e, nc), HASH_THREADS, 0, e.stream>>>((const uint64_t*)cc->values.p, (const uint32_t*)cc->validity.p, nc,
                                                                              cc->dtype == TG_FLOAT64, pkeys, pcap - 1, d_special, allow_nulls, 1,
                                                                              vkeys, vcounts, vcap - 1, d_ex, max_examples, d_ctr);
            TG_CUDA(cudaGetLastError());
            ++launches;
            TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
            TG_CUDA(cudaStreamSynchronize(e.stream));
            if (orphan_rows) fk_orphan_rows64(e, *cc, nc, vkeys, vcap - 1, 0, h.special > 0, orphan, launches);
            const size_t ne = (size_t)std::min<uint64_t>(h.n_examples, (uint64_t)max_examples);
            ex_rows.resize(ne);
            if (ne) TG_CUDA(cudaMemcpy(ex_rows.data(), d_ex, ne * 8, cudaMemcpyDeviceToHost));
        } else if (orphan_rows) {
            fk_orphan_rows64(e, *cc, nc, nullptr, 0, 0, false, orphan, launches);  // no key violates
        }
    } else if (cc->dtype == TG_UTF8 || from_records) {
        const size_t cfp_b = round_up((size_t)nc * 16, 256), cnf_b = round_up((size_t)nc, 256);
        const size_t pfp_b = round_up((size_t)std::max<int64_t>(np, 1) * 16, 256), pnf_b = round_up((size_t)std::max<int64_t>(np, 1), 256);
        const size_t ph_b = pcap * 8;
        const uint64_t vcap = pow2_at_least((uint64_t)nc * 2);  // worst case: every child row violates
        const size_t vh_b = vcap * 8, vc_b = vcap * 4, ex_b = round_up((size_t)std::max(max_examples, 1) * 8, 256);
        uint8_t* scr = e.scratch(cfp_b + cnf_b + pfp_b + pnf_b + 2 * ph_b + 2 * vh_b + vc_b + ex_b + 512);
        uint8_t* q = scr;
        Fp* cfp = (Fp*)q; q += cfp_b;
        uint8_t* cnf = q; q += cnf_b;
        Fp* pfp = (Fp*)q; q += pfp_b;
        uint8_t* pnf = q; q += pnf_b;
        Table128 ptab{(unsigned long long*)q, (unsigned long long*)(q + ph_b), nullptr, pcap - 1}; q += 2 * ph_b;
        Table128 vtab{(unsigned long long*)q, (unsigned long long*)(q + vh_b), (uint32_t*)(q + 2 * vh_b), vcap - 1}; q += 2 * vh_b + vc_b;
        int64_t* d_ex = (int64_t*)q; q += ex_b;
        HashCounters* d_ctr = (HashCounters*)q;
        TG_CUDA(cudaMemsetAsync(ptab.h1, 0xFF, 2 * ph_b, e.stream));
        TG_CUDA(cudaMemsetAsync(vtab.h1, 0xFF, 2 * vh_b, e.stream));
        TG_CUDA(cudaMemsetAsync(vtab.counts, 0, vc_b + ex_b + 512, e.stream));
        if (from_records) {
            fp_unpack_kernel<<<grid_for(e, nc), HASH_THREADS, 0, e.stream>>>((const FpRecord*)cc->values.p, nc, cfp, cnf);
            ++launches;
        } else {
            launches += compute_fingerprints(e, ct, {cc}, cfp, cnf);
        }
        if (np > 0) {
            if (from_records) {
                fp_unpack_kernel<<<grid_for(e, np), HASH_THREADS, 0, e.stream>>>((const FpRecord*)pc->values.p, np, pfp, pnf);
                ++launches;
            } else {
                launches += compute_fingerprints(e, pt, {pc}, pfp, pnf);
            }
            build_set128_kernel<<<grid_for(e, np), HASH_THREADS, 0, e.stream>>>(pfp, pnf, np, ptab);
            ++launches;
        }
        fk_probe128_kernel<<<grid_for(e, nc), HASH_THREADS, 0, e.stream>>>(cfp, cnf, nc, ptab, allow_nulls, 1, vtab, d_ex, max_examples, d_ctr);
        TG_CUDA(cudaGetLastError());
        ++launches;
        TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
        TG_CUDA(cudaStreamSynchronize(e.stream));
        if (orphan_rows) {
            const bool key_viol = h.violations > (allow_nulls ? 0 : h.null_children);
            const Fp128 k{cfp, key_viol ? vtab : Table128{}};
            fk_orphan_rows_kernel<Fp128><<<word_grid(e, nc), HASH_THREADS, 0, e.stream>>>(k, (const uint32_t*)cc->validity.p, nc, orphan);
            TG_CUDA(cudaGetLastError());
            ++launches;
        }
        // (a shard of fingerprint records has no strings to show: counts only, the examples stay empty)
        const size_t ne = from_records ? 0 : (size_t)std::min<uint64_t>(h.n_examples, (uint64_t)max_examples);
        ex_rows.resize(ne);
        if (ne) TG_CUDA(cudaMemcpy(ex_rows.data(), d_ex, ne * 8, cudaMemcpyDeviceToHost));
    } else {
        throw Error(TG_ERR_UNSUPPORTED, "foreign key columns of this type are not supported");
    }
    tm.stop(launches);
    a.u[0] = h.violations;
    a.u[1] = h.distinct_all;
    a.u[2] = h.null_children;
    // examples blob: [count u64][u32 len, bytes]...
    uint64_t cnt = ex_rows.size();
    a.blob.resize(8);
    memcpy(a.blob.data(), &cnt, 8);
    std::sort(ex_rows.begin(), ex_rows.end());
    for (int64_t r : ex_rows) {
        std::string s = row_to_string(e, *cc, r);
        uint32_t L = (uint32_t)s.size();
        size_t o = a.blob.size();
        a.blob.resize(o + 4 + L);
        memcpy(a.blob.data() + o, &L, 4);
        memcpy(a.blob.data() + o + 4, s.data(), L);
    }
}

}  // namespace tg
