// K5 — grouped completeness: GROUP BY g.. -> COUNT(*), COUNT(c), ALL groupings of a plan in ONE pass over the group columns.
//
// Replaces  SELECT g.., COUNT(*), COUNT(c) FROM t GROUP BY g.. [ORDER BY .. LIMIT ..]
//           (analyzers/basic/grouped_completeness.rs:131-176), one query per grouping in the reference.
//
// One fused kernel reads, per row, every DISTINCT group column of the batch once (Utf8: offsets + bytes, fixed width: the
// value; validity bits) and the target columns' validity bits — exactly the algorithmic bytes of SURVEY §8d, nothing is
// materialised per row, and a column shared by several groupings (g0, g1, (g0, g1)) is read and hashed once. A column
// value becomes a 128-bit pair (Utf8 values of at most 8 bytes and fixed-width values carry themselves: no string
// hashing at all); every grouping folds the pairs of its columns into its own fingerprint and counts it in its own
// per-CTA shared-memory table (the common case is a handful to a few thousand groups): a warp first agrees on which
// lanes share a slot (__match_any_sync) so each distinct group costs one shared atomic per warp. A CTA whose table fills
// up spills the row to the grouping's global table directly; at the end every CTA folds its tables into the global
// ones. The first row of every group is kept so the host can fetch the group's key values for the report.
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "engine.hpp"
#include "hash_common.cuh"
#include "ptx.cuh"

namespace tg {

constexpr int GRP_THREADS = 512;
constexpr int GRP_SMEM_BYTES = 222 * 1024;  // dynamic shared memory of the fused kernel, split evenly between the batch's groupings
constexpr int GRP_MAX_PROBE = 24;   // after this many probes the row goes to the global table
constexpr int GRP_MAX_COLS = 8;     // distinct group columns per batch
constexpr int GRP_MAX_JOBS = 4;     // groupings per batch (one kernel launch)
constexpr uint64_t GRP_MAX_GROUPS_DEV = 1u << 20;  // groups per grouping: more is reported as TG_ERR_UNSUPPORTED

struct GrpCol {
    const uint8_t* values;
    const int32_t* offsets;
    const uint32_t* validity;
    int32_t dtype;
    uint32_t job_mask;   // groupings that contain this column
    uint32_t first_mask; // groupings whose FIRST column this is
    uint32_t pad;
};
struct GrpJob {
    const uint32_t* target_validity;
    Table128 gt;  // global table (h1, h2) + parallel arrays below
    unsigned long long* totals;
    unsigned long long* nonnull;
    long long* first_row;
    unsigned long long* n_groups;
};
struct GrpParams {
    GrpCol cols[GRP_MAX_COLS];
    GrpJob jobs[GRP_MAX_JOBS];
    int32_t n_cols, n_jobs;
    int32_t slots[GRP_MAX_JOBS];     // shared-table slots of grouping j (power of two): multi-column groupings get more
    int32_t slot_base[GRP_MAX_JOBS]; // first slot of grouping j in the shared block (24 B per slot)
    int64_t n_rows;
};

constexpr int GRP_ILP = 4;  // rows per thread per iteration: their loads are issued together

// The 128-bit pair a column value contributes. Values that fit carry themselves (x = the bytes, y = a small tag), so two
// different short values can never collide; longer strings are hashed (y has the top bit set: disjoint from the tags).
__device__ __forceinline__ void utf8_pair(const uint8_t* __restrict__ values, int32_t b, int32_t e, uint64_t w0, uint64_t& x, uint64_t& y) {
    const int32_t len = e - b;
    if (len <= 8) {
        x = w0;
        y = (uint64_t)len;
        return;
    }
    x = 0x736f6d6570736575ull ^ (uint64_t)len;
    y = 0x646f72616e646f6dull + (uint64_t)len * 0x100000001b3ull;
    for (int32_t p = b; p < e; p += 8) {
        const uint64_t ww = p == b ? w0 : load_upto8(values, p, min(8, e - p));
        x = (x ^ ww) * 0x9fb21c651e98df25ull;
        x ^= x >> 29;
        y = (y + ww) * 0xc2b2ae3d27d4eb4full;
        y ^= y >> 31;
    }
    y |= 0x8000000000000000ull;
}

// Once a grouping holds more than GRP_MAX_GROUPS_DEV groups (the most the host reports), it stops counting: the result
// is the "more than 1048576 groups" error anyway, and the global table (up to 4 x GRP_MAX_GROUPS_DEV slots, at least
// 2 x n) stays far from full, where upsert128 would probe without end. The overshoot is bounded by the threads in flight.
__device__ __noinline__ void global_count(const GrpJob& J, Fp f, unsigned long long tot, unsigned long long nn, long long first) {
    if (*reinterpret_cast<volatile unsigned long long*>(J.n_groups) > GRP_MAX_GROUPS_DEV) return;
    bool created;
    const uint64_t slot = upsert128(J.gt, f, created);
    if (created) atomicAdd(J.n_groups, 1ull);
    if (tot) atomicAdd(&J.totals[slot], tot);
    if (nn) atomicAdd(&J.nonnull[slot], nn);
    atomicMin(&J.first_row[slot], first);
}

// find-or-insert (a, b) in a grouping's shared table; returns the slot or -1 when the probe limit is hit. Kept out of
// line: it is called GRP_ILP x groupings times per iteration and inlining every copy overflows the instruction cache.
// Only the thread that claimed the first word writes the second one; others wait for it (as upsert128 does). Two groups
// may share the first word (Utf8 values that differ in trailing NUL bytes only, or a key whose bits equal NULL_TAG1 next
// to a NULL): a second thread must not take the slot before the claimer has published which group it holds.
__device__ __noinline__ int smem_upsert(unsigned long long* s_h1, unsigned long long* s_h2, uint32_t mask, unsigned long long a,
                                        unsigned long long b, bool& created) {
    created = false;
    uint32_t s = (uint32_t)(a ^ (b >> 32)) & mask;
    for (int probe = 0; probe < GRP_MAX_PROBE; ++probe, s = (s + 1) & mask) {
        unsigned long long v = s_h1[s];
        if (v == EMPTY64) {
            v = atomicCAS(&s_h1[s], EMPTY64, a);
            if (v == EMPTY64) {  // claimed: publish the second word (never EMPTY64: the caller maps it to 0)
                atomicExch(&s_h2[s], b);
                created = true;
                return (int)s;
            }
        }
        if (v == a) {
            unsigned long long w;
            do {
                w = *reinterpret_cast<volatile unsigned long long*>(&s_h2[s]);
            } while (w == EMPTY64);
            if (w == b) return (int)s;  // a different second word: another group
        }
    }
    return -1;
}

// shared memory of grouping j: [h1: slots x 8][h2: slots x 8][tot: slots x 4][nn: slots x 4]
template <int NJ>
__global__ void __launch_bounds__(GRP_THREADS, 1) group_count_fused_kernel(const __grid_constant__ GrpParams P) {
    extern __shared__ __align__(16) unsigned long long grp_smem[];
    unsigned long long* s_h1[NJ];
    unsigned long long* s_h2[NJ];
    uint32_t* s_tot[NJ];
    uint32_t* s_nn[NJ];
    uint32_t smask[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const int slots = P.slots[j];
        unsigned long long* base = grp_smem + (size_t)P.slot_base[j] * 3;
        s_h1[j] = base;
        s_h2[j] = base + slots;
        s_tot[j] = reinterpret_cast<uint32_t*>(base + 2 * slots);
        s_nn[j] = s_tot[j] + slots;
        smask[j] = (uint32_t)slots - 1u;
        for (int s = threadIdx.x; s < slots; s += GRP_THREADS) {
            s_h1[j][s] = EMPTY64;
            s_h2[j][s] = EMPTY64;
            s_tot[j][s] = 0;
            s_nn[j][s] = 0;
        }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    for (int64_t base0 = (int64_t)blockIdx.x * GRP_THREADS * GRP_ILP; base0 < P.n_rows; base0 += (int64_t)gridDim.x * GRP_THREADS * GRP_ILP) {
        int64_t row[GRP_ILP];
        bool act[GRP_ILP];
        Fp fps[NJ][GRP_ILP];
#pragma unroll
        for (int k = 0; k < GRP_ILP; ++k) {
            row[k] = base0 + (int64_t)k * GRP_THREADS + threadIdx.x;
            act[k] = row[k] < P.n_rows;
        }
#pragma unroll
        for (int j = 0; j < NJ; ++j)
#pragma unroll
            for (int k = 0; k < GRP_ILP; ++k) fps[j][k] = Fp{0, 0};
        // ---- every distinct group column once: loads of the GRP_ILP rows go out in waves (validity + offsets or values,
        // then the first 8 key bytes) before anything is hashed; the column's pair is folded into every grouping it is in
        for (int i = 0; i < P.n_cols; ++i) {
            const GrpCol& c = P.cols[i];
            bool valid[GRP_ILP];
            uint64_t x[GRP_ILP], y[GRP_ILP];
#pragma unroll
            for (int k = 0; k < GRP_ILP; ++k) valid[k] = act[k] && row_valid(c.validity, row[k]);
            if (c.dtype == TG_UTF8) {
                int32_t b[GRP_ILP], e[GRP_ILP];
                uint64_t w[GRP_ILP];
#pragma unroll
                for (int k = 0; k < GRP_ILP; ++k) {
                    b[k] = valid[k] ? __ldg(c.offsets + row[k]) : 0;
                    e[k] = valid[k] ? __ldg(c.offsets + row[k] + 1) : 0;
                }
#pragma unroll
                for (int k = 0; k < GRP_ILP; ++k) w[k] = e[k] > b[k] ? load_upto8(c.values, b[k], min(8, e[k] - b[k])) : 0ull;
#pragma unroll
                for (int k = 0; k < GRP_ILP; ++k) {
                    if (valid[k]) utf8_pair(c.values, b[k], e[k], w[k], x[k], y[k]);
                }
            } else {
#pragma unroll
                for (int k = 0; k < GRP_ILP; ++k) {
                    x[k] = 0;
                    y[k] = 0x10ull + (uint64_t)c.dtype;  // fixed-width tag (Utf8 lengths use 0..8)
                    if (!valid[k]) continue;
                    const int64_t r = row[k];
                    switch (c.dtype) {
                        case TG_INT64: x[k] = __ldg(reinterpret_cast<const unsigned long long*>(c.values) + r); break;
                        case TG_FLOAT64: x[k] = canon_f64(__ldg(reinterpret_cast<const unsigned long long*>(c.values) + r)); break;
                        case TG_INT32: x[k] = (uint64_t)(int64_t)__ldg(reinterpret_cast<const int32_t*>(c.values) + r); break;
                        case TG_FLOAT32: x[k] = canon_f64((uint64_t)__double_as_longlong((double)__ldg(reinterpret_cast<const float*>(c.values) + r))); break;
                        default: x[k] = (__ldg(reinterpret_cast<const uint32_t*>(c.values) + (r >> 5)) >> (r & 31)) & 1u; break;  // TG_BOOL
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < GRP_ILP; ++k) {
                if (!valid[k]) {
                    x[k] = NULL_TAG1;
                    y[k] = NULL_TAG2;
                }
            }
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                if (!((c.job_mask >> j) & 1u)) continue;
                const bool first = (c.first_mask >> j) & 1u;
#pragma unroll
                for (int k = 0; k < GRP_ILP; ++k) fp_combine(fps[j][k], x[k], y[k], first);
            }
        }
        // ---- count: per grouping, per row
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const GrpJob& J = P.jobs[j];
#pragma unroll
            for (int k = 0; k < GRP_ILP; ++k) {
                const bool ok = act[k] && row_valid(J.target_validity, row[k]);
                int slot = -1;  // shared slot, or -1: not active / spilled
                if (act[k]) {
                    // EMPTY64 is the shared table's vacancy marker in both words
                    const unsigned long long a = fps[j][k].h1 == EMPTY64 ? 0ull : fps[j][k].h1, b = fps[j][k].h2 == EMPTY64 ? 0ull : fps[j][k].h2;
                    bool created;
                    slot = smem_upsert(s_h1[j], s_h2[j], smask[j], a, b, created);
                    // a new group of this CTA registers itself (and a representative row) in the global table right away;
                    // a row that finds the shared table full is counted there directly
                    if (slot < 0) global_count(J, fps[j][k], 1ull, ok ? 1ull : 0ull, (long long)row[k]);
                    else if (created) global_count(J, fps[j][k], 0ull, 0ull, (long long)row[k]);
                }
                // one shared atomic per distinct slot per warp
                const unsigned peers = __match_any_sync(0xffffffffu, slot);
                const unsigned ok_peers = __ballot_sync(0xffffffffu, ok) & peers;
                if (slot >= 0 && lane == __ffs(peers) - 1) {
                    atomicAdd(&s_tot[j][slot], (uint32_t)__popc(peers));
                    const int c = __popc(ok_peers);
                    if (c) atomicAdd(&s_nn[j][slot], (uint32_t)c);
                }
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        for (int i = threadIdx.x; i < P.slots[j]; i += GRP_THREADS) {
            if (s_tot[j][i] == 0) continue;
            // EMPTY64 was mapped to 0 above exactly like upsert128 maps it, so the pair can be handed over as is
            global_count(P.jobs[j], Fp{s_h1[j][i], s_h2[j][i]}, s_tot[j][i], s_nn[j][i], INT64_MAX);
        }
    }
}

// =====================================================================================================================
// Fast path: per-CTA column dictionaries. Group columns are low-cardinality almost by definition (the reference caps a
// grouping at max_groups = 10 000, analyzers/grouped.rs:36), so a CTA keeps, per distinct group column, a small
// shared-memory dictionary value -> slot. A value is identified EXACTLY: fixed-width values and Utf8 values of at most 8
// bytes by their bits plus a tag (length / type / NULL), longer strings by a 128-bit hash pair. Per row a column costs
// one cheap 32-bit hash and one probe; a single-column grouping counts straight into counters parallel to the
// dictionary, a 2- / 3-column grouping keys a second shared table with the packed slot numbers (10 bits each). No
// 64-bit multiply chains, no per-grouping string hashing. At the end a CTA publishes its dictionary entries to the
// column's global dictionary (a 128-bit table: the global slot is the value's code), adds its counters at those codes
// and folds its composite tables into the grouping's global table keyed by the packed global codes. A CTA whose
// dictionary or composite table overflows raises a flag and the host re-runs the batch through the generic
// fingerprint kernel above.
// =====================================================================================================================
#ifndef TG_GD_THREADS
#define TG_GD_THREADS 1024
#define TG_GD_ILP 4
#endif
constexpr int GD_THREADS = TG_GD_THREADS, GD_ILP = TG_GD_ILP;
constexpr int GD_DICT = 1024;       // dictionary slots per column per CTA (10-bit local codes)
constexpr int GD_MAX_COLS = 4, GD_MAX_JOBS = 4;
constexpr int GD_PROBE = 16;
constexpr int GD_CODE_BITS = 21;    // global dictionary slots per column <= 2^21: three codes fit one 64-bit composite key
constexpr size_t GD_CTA_ROWS_BYTES = (size_t)256 * 8192 * 4;  // per composite grouping: up to 256 CTAs x 8192 slots x 4 bytes
constexpr uint32_t GD_TAG_NULL = 0x40u, GD_TAG_LONG = 0x80u, GD_BUSY = 0xFFFFFFFFu;

struct GdCol {
    const uint8_t* values;
    const int32_t* offsets;
    const uint32_t* validity;
    int32_t dtype;
    uint32_t smem_off;     // byte offset of the column's dictionary in dynamic shared memory
    Table128 dict;         // global dictionary (h1, h2); the slot is the value's global code
    long long* first_row;  // a representative row per global slot
};
struct GdJob {
    const uint32_t* target_validity;
    int32_t n_cols;
    int32_t col[3];
    uint32_t smem_off;       // single-column: counters [tot GD_DICT][nul GD_DICT]; composite: [key S][tot S][nul S]
    uint32_t comp_slots;     // composite: S (power of two); single-column: 0
    int32_t derived_from;    // >= 0: this single-column grouping is a marginal of that composite job (same target): not
    int32_t derived_pos;     // counted per row; its column's code sits at bits [10 * derived_pos ..) of the composite key
    // global state. single-column: totals / nonnull indexed by the column's global code. composite: 64-bit key table.
    unsigned long long* totals;
    unsigned long long* nonnull;
    unsigned long long* ckeys;  // composite keys (EMPTY64 = vacant)
    long long* crow;            // composite: representative row
    uint32_t* cta_rows;         // composite: [CTA][comp_slots] representative row of the CTA's table entry (kept out of shared memory)
    uint64_t cmask;
};
// staging ring of the tile kernel: per stage, per column the pieces below (byte offsets inside a stage; 0xFFFFFFFF = none)
struct GdStageCol {
    uint32_t main_off;   // Utf8: offsets of the tile's rows (+1); fixed width: the values
    uint32_t bytes_off;  // Utf8: the tile's string bytes, from the 16-byte boundary below its first byte
    uint32_t bytes_cap;  // Utf8: room for them (a tile with more is read from global memory)
    uint32_t val_off;    // validity words
};
struct GdParams {
    GdCol cols[GD_MAX_COLS];
    GdJob jobs[GD_MAX_JOBS];
    int32_t n_cols, n_jobs;
    int64_t n_rows;
    unsigned int* overflow;
    // tile kernel only
    GdStageCol st[GD_MAX_COLS];
    uint32_t st_target[GD_MAX_JOBS];  // target validity words of job j inside a stage (shared by jobs with one target)
    uint32_t ring_off, stage_bytes, n_stages;
    uint32_t tv_copy_mask;            // bit j: job j is the first user of its target piece (the producer copies it once)
};

// dictionary of one column in shared memory: 16-byte entries {x.lo, x.hi, state, row} — a probe is ONE 128-bit shared
// load — and the second hash word of long strings in a parallel array (only read for entries tagged GD_TAG_LONG)
struct GdDict {
    uint4* ent;              // [GD_DICT] .x/.y value bits (first hash word), .z state: 0 vacant, GD_BUSY being written, else
                             // the tag (never 0), .w a row holding the value; after the publish step: the global code
    unsigned long long* y;   // [GD_DICT] second hash word of long strings (0 otherwise)
};
__device__ __forceinline__ GdDict gd_dict(uint8_t* smem, uint32_t off) {
    GdDict d;
    d.ent = reinterpret_cast<uint4*>(smem + off);
    d.y = reinterpret_cast<unsigned long long*>(smem + off + GD_DICT * 16);
    return d;
}
constexpr uint32_t GD_DICT_BYTES = GD_DICT * 24;

__device__ __forceinline__ uint32_t gd_hash(uint64_t x, uint32_t tag) {
    uint32_t h = (uint32_t)x * 0x9E3779B1u ^ (uint32_t)(x >> 32) * 0x85EBCA77u ^ tag * 0xC2B2AE3Du;
    h ^= h >> 15;
    return (h * 0x2C1B3C6Du) >> 22;  // GD_DICT = 1024 slots
}
static_assert(GD_DICT == 1024, "gd_hash keeps the top 10 bits");

__device__ __forceinline__ uint4 lds128_volatile(const uint4* p) {
    uint4 r;
    asm volatile("ld.volatile.shared.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "r"((uint32_t)__cvta_generic_to_shared(p)));
    return r;
}

__device__ __noinline__ ulonglong2 gd_long_pair(const uint8_t* __restrict__ values, int32_t b, int32_t e, uint64_t w0) {
    uint64_t hx, hy;
    utf8_pair(values, b, e, w0, hx, hy);
    return make_ulonglong2(hx, hy);
}

// find-or-insert, the general case (first-probe hits are answered inline by the caller); returns the slot, or -1 when the
// probe limit is hit (dictionary too small for this column)
__device__ __noinline__ int gd_lookup_slow(const GdDict d, uint32_t s, uint64_t x, uint64_t y, uint32_t tag, uint32_t row) {
    for (int probe = 0; probe < GD_PROBE; ++probe, s = (s + 1) & (GD_DICT - 1)) {
        uint32_t* state = &d.ent[s].z;
        while (true) {
            uint32_t st = *reinterpret_cast<volatile uint32_t*>(state);
            if (st == 0u) {
                st = atomicCAS(state, 0u, GD_BUSY);
                if (st == 0u) {  // claimed: fill, then publish the tag
                    d.ent[s].x = (uint32_t)x;
                    d.ent[s].y = (uint32_t)(x >> 32);
                    d.ent[s].w = row;
                    d.y[s] = y;
                    __threadfence_block();
                    atomicExch(state, tag);
                    return (int)s;
                }
            }
            if (st == GD_BUSY) continue;  // another thread is writing the entry: look again
            const uint4 e = lds128_volatile(&d.ent[s]);
            if (st == tag && e.x == (uint32_t)x && e.y == (uint32_t)(x >> 32) &&
                (tag != GD_TAG_LONG || *reinterpret_cast<volatile unsigned long long*>(&d.y[s]) == y))
                return (int)s;
            break;  // another value lives here
        }
    }
    return -1;
}

// find-or-insert of a packed composite key in a job's shared table [key S][tot S][nul S] (+ the entry's row in global memory)
__device__ __noinline__ int gd_comp_slow(uint32_t* jb, uint32_t* cta_rows, uint32_t S, uint32_t s, uint32_t key, uint32_t row,
                                         uint32_t* n_entries = nullptr) {
    for (int probe = 0; probe < GD_PROBE; ++probe, s = (s + 1) & (S - 1)) {
        uint32_t v = *reinterpret_cast<volatile uint32_t*>(&jb[s]);
        if (v == 0xFFFFFFFFu) {
            v = atomicCAS(&jb[s], 0xFFFFFFFFu, key);
            if (v == 0xFFFFFFFFu) {
                cta_rows[s] = row;  // representative row, the CTA's own slice (read by this CTA after a barrier only)
                if (n_entries) atomicAdd(n_entries, 1u);
                return (int)s;
            }
        }
        if (v == key) return (int)s;
    }
    return -1;
}

__device__ __forceinline__ uint64_t upsert64(unsigned long long* keys, uint64_t mask, uint64_t k) {
    uint64_t s = fmix64(k) & mask;
    while (true) {
        const unsigned long long prev = atomicCAS(&keys[s], EMPTY64, (unsigned long long)k);
        if (prev == EMPTY64 || prev == k) return s;
        s = (s + 1) & mask;
    }
}

// End of a counting kernel (either variant): marginal groupings summed out of the composite tables, local dictionary
// slots published as global codes, counters folded into the global tables. `late_zero`: the derived groupings' counters
// alias memory the main loop used (the staging ring) and are cleared here first.
template <int NC>
__device__ __forceinline__ void gd_fold(const GdParams& P, uint8_t* gd_smem, bool overflow, bool late_zero) {
    const int GDT = blockDim.x;
    if (overflow) atomicExch(P.overflow, 1u);
    __syncthreads();
    if (late_zero) {
        for (int j = 0; j < P.n_jobs; ++j) {
            const GdJob& J = P.jobs[j];
            if (J.derived_from < 0) continue;
            uint32_t* jb = reinterpret_cast<uint32_t*>(gd_smem + J.smem_off);
            for (int s = threadIdx.x; s < 2 * GD_DICT; s += GDT) jb[s] = 0u;
        }
        __syncthreads();
    }
    // ---- marginals: a derived single-column grouping gets its counters from the composite table it is a marginal of
    for (int j = 0; j < P.n_jobs; ++j) {
        const GdJob& J = P.jobs[j];
        if (J.derived_from < 0) continue;
        const GdJob& Q = P.jobs[J.derived_from];
        const uint32_t* qb = reinterpret_cast<const uint32_t*>(gd_smem + Q.smem_off);
        uint32_t* jb = reinterpret_cast<uint32_t*>(gd_smem + J.smem_off);
        const uint32_t S = Q.comp_slots;
        for (uint32_t s = threadIdx.x; s < S; s += GDT) {
            const uint32_t key = qb[s];
            if (key == 0xFFFFFFFFu) continue;
            const uint32_t code = (key >> (10 * J.derived_pos)) & 1023u;
            atomicAdd(&jb[code], qb[S + s]);
            if (qb[2 * S + s]) atomicAdd(&jb[GD_DICT + code], qb[2 * S + s]);
        }
    }
    // ---- publish the dictionaries: local slot -> global code (kept in ent.w), representative row -> first_row
    for (int c = 0; c < NC; ++c) {
        const GdCol& C = P.cols[c];
        const GdDict d = gd_dict(gd_smem, C.smem_off);
        for (int s = threadIdx.x; s < GD_DICT; s += GDT) {
            const uint4 en = d.ent[s];
            const uint32_t tag = en.z;
            if (tag == 0u) continue;
            const uint64_t x = (uint64_t)en.x | ((uint64_t)en.y << 32);
            Fp f{0, 0};
            fp_combine(f, x ^ ((uint64_t)tag << 56), d.y[s] + tag, true);
            // exact for short values: fp_combine(first) applies two bijections, to (x ^ tag << 56) and to (y + tag); the tag's
            // bits 56.. can only meet value bits for 8-byte values, whose tag (9 / a type tag) is fixed per column
            bool created;
            const uint64_t g = upsert128(C.dict, f, created);
            atomicMin(&C.first_row[g], (long long)en.w);
            d.ent[s].w = (uint32_t)g;
        }
    }
    __syncthreads();
    for (int j = 0; j < P.n_jobs; ++j) {
        const GdJob& J = P.jobs[j];
        uint32_t* jb = reinterpret_cast<uint32_t*>(gd_smem + J.smem_off);
        if (J.comp_slots == 0) {
            const GdDict d = gd_dict(gd_smem, P.cols[J.col[0]].smem_off);
            for (int s = threadIdx.x; s < GD_DICT; s += GDT) {
                const uint32_t t = jb[s];
                if (!t || d.ent[s].z == 0u) continue;  // (a counter without an entry: rows parked at slot 0 after an overflow)
                const uint32_t g = d.ent[s].w;
                atomicAdd(&J.totals[g], (unsigned long long)t);
                if (t != jb[GD_DICT + s]) atomicAdd(&J.nonnull[g], (unsigned long long)(t - jb[GD_DICT + s]));
            }
        } else {
            const uint32_t S = J.comp_slots;
            const GdDict d0 = gd_dict(gd_smem, P.cols[J.col[0]].smem_off), d1 = gd_dict(gd_smem, P.cols[J.col[1]].smem_off);
            const GdDict d2 = gd_dict(gd_smem, P.cols[J.col[J.n_cols > 2 ? 2 : 0]].smem_off);
            for (uint32_t s = threadIdx.x; s < S; s += GDT) {
                const uint32_t key = jb[s];
                if (key == 0xFFFFFFFFu) continue;
                uint64_t K = (uint64_t)d0.ent[key & 1023u].w | ((uint64_t)d1.ent[(key >> 10) & 1023u].w << GD_CODE_BITS);
                if (J.n_cols > 2) K |= (uint64_t)d2.ent[(key >> 20) & 1023u].w << (2 * GD_CODE_BITS);
                const uint64_t g = upsert64(J.ckeys, J.cmask, K);
                const uint32_t t = jb[S + s], nl = jb[2 * S + s];
                atomicAdd(&J.totals[g], (unsigned long long)t);
                if (t != nl) atomicAdd(&J.nonnull[g], (unsigned long long)(t - nl));
                atomicMin(&J.crow[g], (long long)J.cta_rows[(size_t)blockIdx.x * S + s]);
            }
        }
    }
}

// A warp owns 32 * GD_ILP consecutive rows per iteration (lane l: rows l, 32 + l, ...): validity words are one broadcast
// load per 32 rows, offsets and string bytes are read coalesced, and the GD_ILP independent rows of a lane keep that many
// dependent load chains (offset -> bytes -> dictionary) in flight. Per row: one inline first-probe hit per distinct group
// column (a 128-bit shared load and a compare), the local codes of the row packed 10 bits per column, one counter update
// per COUNTED grouping (a single-column grouping that is a marginal of a composite grouping over the same target is not
// counted per row: the CTA derives it from the composite table before folding), NULL targets counted instead of non-NULL
// ones (they are the rare case).
template <int NC>
__global__ void __launch_bounds__(GD_THREADS, 1) group_count_dict_kernel(const __grid_constant__ GdParams P) {
    extern __shared__ __align__(16) uint8_t gd_smem[];
    // ---- clear the dictionaries and the job tables
    for (int c = 0; c < NC; ++c) {
        const GdDict d = gd_dict(gd_smem, P.cols[c].smem_off);
        for (int s = threadIdx.x; s < GD_DICT; s += GD_THREADS) d.ent[s].z = 0u;
    }
    for (int j = 0; j < P.n_jobs; ++j) {
        const GdJob& J = P.jobs[j];
        uint32_t* base = reinterpret_cast<uint32_t*>(gd_smem + J.smem_off);
        if (J.comp_slots == 0) {
            for (int s = threadIdx.x; s < 2 * GD_DICT; s += GD_THREADS) base[s] = 0u;
        } else {
            for (uint32_t s = threadIdx.x; s < J.comp_slots; s += GD_THREADS) {
                base[s] = 0xFFFFFFFFu;
                base[J.comp_slots + s] = 0u;
                base[2 * J.comp_slots + s] = 0u;
            }
        }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    bool overflow = false;
    for (int64_t base0 = (int64_t)blockIdx.x * GD_THREADS * GD_ILP; base0 < P.n_rows; base0 += (int64_t)gridDim.x * GD_THREADS * GD_ILP) {
        const int64_t wrow0 = base0 + (int64_t)warp * 32 * GD_ILP;  // first row of the warp (a multiple of 32)
        if (wrow0 >= P.n_rows) continue;
        // Rows past the end are clamped to the last row for every load (in bounds, branch-free) and dropped at the counters.
        uint32_t row[GD_ILP];  // n_rows < 2^32 (checked by the host)
        uint32_t packed[GD_ILP];   // local code of column c in bits [10c ..), c < 3;
        uint32_t packed3[GD_ILP];  // the 4th column's code apart
        const uint32_t last_row = (uint32_t)(P.n_rows - 1);
        const int64_t word0 = wrow0 >> 5;                       // warp-uniform validity word of k = 0
        const int64_t last_word = (P.n_rows - 1) >> 5;
#pragma unroll
        for (int k = 0; k < GD_ILP; ++k) {
            row[k] = min((uint32_t)(wrow0 + k * 32 + lane), last_row);
            packed[k] = 0;
            packed3[k] = 0;
        }
        // ---- every distinct group column once
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const GdCol& C = P.cols[c];
            const GdDict d = gd_dict(gd_smem, C.smem_off);
            uint32_t vbit[GD_ILP];
            uint64_t x[GD_ILP], y[GD_ILP];
            uint32_t tag[GD_ILP];
#pragma unroll
            for (int k = 0; k < GD_ILP; ++k) {
                const uint32_t vw = C.validity ? __ldg(C.validity + min(word0 + k, last_word)) : 0xffffffffu;
                vbit[k] = (vw >> (row[k] & 31u)) & 1u;
                y[k] = 0;
            }
            if (C.dtype == TG_UTF8) {
                // branch-free for strings of at most 8 bytes: both offsets, the two aligned 8-byte words around the start (the
                // value buffer is padded: the over-read stays in bounds), a 128-bit funnel shift and a length mask
                int32_t b[GD_ILP], len[GD_ILP];
                uint2 w0[GD_ILP], w1[GD_ILP];
#pragma unroll
                for (int k = 0; k < GD_ILP; ++k) {
                    const int32_t* op = C.offsets + row[k];
                    b[k] = __ldg(op);
                    len[k] = __ldg(op + 1) - b[k];
                }
#pragma unroll
                for (int k = 0; k < GD_ILP; ++k) {
                    const uint2* vp = reinterpret_cast<const uint2*>(C.values + ((uint32_t)b[k] & ~7u));
                    w0[k] = __ldg(vp);
                    w1[k] = __ldg(vp + 1);
                }
                bool any_long = false;
#pragma unroll
                for (int k = 0; k < GD_ILP; ++k) {
                    const uint32_t sh = ((uint32_t)b[k] & 7u) * 8u, sl = sh & 31u;
                    const bool up = sh >= 32u;
                    const uint32_t A = up ? w0[k].y : w0[k].x, Bw = up ? w1[k].x : w0[k].y, Cw = up ? w1[k].y : w1[k].x;
                    const uint32_t lo = __funnelshift_r(A, Bw, sl), hi = __funnelshift_r(Bw, Cw, sl);
                    const uint32_t nb = (uint32_t)min(len[k], 8) * 8u;  // bits kept
                    const uint32_t mlo = nb >= 32u ? 0xffffffffu : ((1u << nb) - 1u);
                    const uint32_t mhi = nb >= 64u ? 0xffffffffu : (nb > 32u ? ((1u << (nb - 32u)) - 1u) : 0u);
                    x[k] = (uint64_t)(lo & mlo) | ((uint64_t)(hi & mhi) << 32);
                    tag[k] = (uint32_t)len[k] + 1u;  // 1..9
                    any_long |= len[k] > 8 && vbit[k];
                }
                if (__any_sync(0xffffffffu, any_long)) {  // longer strings: identified by a 128-bit hash pair
#pragma unroll
                    for (int k = 0; k < GD_ILP; ++k) {
                        if (len[k] > 8 && vbit[k]) {
                            const ulonglong2 h2 = gd_long_pair(C.values, b[k], b[k] + len[k], x[k]);
                            x[k] = h2.x;
                            y[k] = h2.y;
                            tag[k] = GD_TAG_LONG;
                        }
                    }
                }
            } else {
#pragma unroll
                for (int k = 0; k < GD_ILP; ++k) {
                    tag[k] = 0x10u + (uint32_t)C.dtype;
                    const int64_t r = row[k];
                    switch (C.dtype) {
                        case TG_INT64: x[k] = __ldg(reinterpret_cast<const unsigned long long*>(C.values) + r); break;
                        case TG_FLOAT64: x[k] = canon_f64(__ldg(reinterpret_cast<const unsigned long long*>(C.values) + r)); break;
                        case TG_INT32: x[k] = (uint64_t)(int64_t)__ldg(reinterpret_cast<const int32_t*>(C.values) + r); break;
                        case TG_FLOAT32: x[k] = canon_f64((uint64_t)__double_as_longlong((double)__ldg(reinterpret_cast<const float*>(C.values) + r))); break;
                        default: x[k] = (__ldg(reinterpret_cast<const uint32_t*>(C.values) + (r >> 5)) >> (r & 31)) & 1u; break;  // TG_BOOL
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < GD_ILP; ++k) {
                if (!vbit[k]) {
                    x[k] = 0;
                    y[k] = 0;
                    tag[k] = GD_TAG_NULL;
                }
                int s = (int)gd_hash(x[k], tag[k]);
                // hits are answered inline (linear probing at a load of <= 20 %: one or two probes); vacant or busy entries
                // and long strings (second hash word) go through the out-of-line find-or-insert
                bool hit = false;
#pragma unroll 1
                for (int probe = 0; probe < GD_PROBE; ++probe) {
                    const uint4 en = lds128_volatile(&d.ent[s]);
                    hit = en.z == tag[k] && en.x == (uint32_t)x[k] && en.y == (uint32_t)(x[k] >> 32);
                    if (hit || en.z == 0u || en.z == GD_BUSY) break;
                    s = (s + 1) & (GD_DICT - 1);
                }
                if (!hit || tag[k] == GD_TAG_LONG) s = gd_lookup_slow(d, (uint32_t)s, x[k], y[k], tag[k], row[k]);
                if (s < 0) {
                    overflow = true;
                    s = 0;
                }
                if (c < 3) packed[k] |= (uint32_t)s << (10 * c);
                else packed3[k] = (uint32_t)s;
            }
        }
        // ---- count: per counted grouping, per row
        for (int j = 0; j < P.n_jobs; ++j) {
            const GdJob& J = P.jobs[j];
            if (J.derived_from >= 0) continue;
            uint32_t* jb = reinterpret_cast<uint32_t*>(gd_smem + J.smem_off);
            const uint32_t S = J.comp_slots;
            uint32_t* tot = S ? jb + S : jb;
            uint32_t* nul = S ? jb + 2 * S : jb + GD_DICT;
            const int c0 = J.col[0], c1 = J.col[1], c2 = J.col[2];
#pragma unroll
            for (int k = 0; k < GD_ILP; ++k) {
                const uint32_t tw = J.target_validity ? __ldg(J.target_validity + min(word0 + k, last_word)) : 0xffffffffu;
                const uint32_t s0 = c0 < 3 ? (packed[k] >> (10 * c0)) & 1023u : packed3[k];
                int cs = (int)s0;
                if (S) {
                    const uint32_t s1 = c1 < 3 ? (packed[k] >> (10 * c1)) & 1023u : packed3[k];
                    const uint32_t s2 = J.n_cols > 2 ? (c2 < 3 ? (packed[k] >> (10 * c2)) & 1023u : packed3[k]) : 0u;
                    const uint32_t key = s0 | (s1 << 10) | (s2 << 20);
                    uint32_t h = key * 0x9E3779B1u;
                    h ^= h >> 15;
                    uint32_t s = h & (S - 1);
                    bool hit = false;
#pragma unroll 1
                    for (int probe = 0; probe < GD_PROBE; ++probe) {
                        const uint32_t v = *reinterpret_cast<volatile uint32_t*>(&jb[s]);
                        hit = v == key;
                        if (hit || v == 0xFFFFFFFFu) break;
                        s = (s + 1) & (S - 1);
                    }
                    cs = hit ? (int)s : gd_comp_slow(jb, J.cta_rows + (size_t)blockIdx.x * S, S, s, key, row[k]);
                    if (cs < 0) overflow = true;
                }
                if (wrow0 + k * 32 + lane >= P.n_rows) cs = -1;  // a clamped row past the end
                // one shared atomic per distinct counter per warp (measured: plain per-lane shared atomics are 2x slower here)
                const unsigned peers = __match_any_sync(0xffffffffu, cs);
                if (cs >= 0) {
                    if (lane == __ffs(peers) - 1) atomicAdd(&tot[cs], (uint32_t)__popc(peers));
                    if (!((tw >> lane) & 1u)) atomicAdd(&nul[cs], 1u);
                }
            }
        }
    }
    gd_fold<NC>(P, gd_smem, overflow, false);
}

// =====================================================================================================================
// Tile variant of the dictionary kernel (the one that normally runs): a producer warp stages every tile of GT_ROWS rows —
// offsets, the tile's string bytes, fixed-width values, validity words of the group columns and of the targets — in a
// shared-memory ring with TMA bulk copies (cp.async.bulk + mbarrier complete_tx), 24 consumer warps take one row per
// lane from shared memory. A row's dependent chain offset -> bytes -> dictionary runs at shared-memory latency, nothing
// is unrolled (small code, no register pressure), and every byte crosses HBM -> SM once. CTAs own contiguous tile
// ranges so a tile's last offset is the next tile's first; the producer fetches 32 tile boundaries per round trip.
// =====================================================================================================================
constexpr int GT_CONSUMER_WARPS = 24, GT_THREADS = (GT_CONSUMER_WARPS + 1) * 32, GT_ROWS = GT_CONSUMER_WARPS * 32;
constexpr int GT_MAX_STAGES = 4;
#ifndef TG_GT_DIRECT_GROUPS
#define TG_GT_DIRECT_GROUPS 256
#endif
constexpr uint32_t GT_DIRECT_GROUPS = TG_GT_DIRECT_GROUPS;  // composite groups in the CTA's table from which the counters are bumped per lane

template <int NC>
__global__ void __launch_bounds__(GT_THREADS, 1) group_count_tile_kernel(const __grid_constant__ GdParams P) {
    extern __shared__ __align__(16) uint8_t gd_smem[];
    __shared__ __align__(8) uint64_t full[GT_MAX_STAGES], empty[GT_MAX_STAGES];
    __shared__ uint32_t s_byte_base[GT_MAX_STAGES][GD_MAX_COLS];  // absolute byte offset staged at bytes_off; 0xFFFFFFFF: not staged
    __shared__ uint32_t s_comp_entries[GD_MAX_JOBS];              // composite groups this CTA has met so far
    if (threadIdx.x < GD_MAX_JOBS) s_comp_entries[threadIdx.x] = 0u;
    for (int c = 0; c < NC; ++c) {
        const GdDict d = gd_dict(gd_smem, P.cols[c].smem_off);
        for (int s = threadIdx.x; s < GD_DICT; s += GT_THREADS) d.ent[s].z = 0u;
    }
    for (int j = 0; j < P.n_jobs; ++j) {
        const GdJob& J = P.jobs[j];
        if (J.derived_from >= 0) continue;  // cleared by the fold (their counters alias the ring)
        uint32_t* base = reinterpret_cast<uint32_t*>(gd_smem + J.smem_off);
        if (J.comp_slots == 0) {
            for (int s = threadIdx.x; s < 2 * GD_DICT; s += GT_THREADS) base[s] = 0u;
        } else {
            for (uint32_t s = threadIdx.x; s < J.comp_slots; s += GT_THREADS) {
                base[s] = 0xFFFFFFFFu;
                base[J.comp_slots + s] = 0u;
                base[2 * J.comp_slots + s] = 0u;
            }
        }
    }
    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < P.n_stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], GT_CONSUMER_WARPS);
        }
        mbar_fence_init();
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n_tiles = (P.n_rows + GT_ROWS - 1) / GT_ROWS;
    const int64_t t_begin = n_tiles * blockIdx.x / gridDim.x, t_end = n_tiles * (blockIdx.x + 1) / gridDim.x;
    uint8_t* ring = gd_smem + P.ring_off;
    bool overflow = false;
    if (warp == GT_CONSUMER_WARPS) {
        // ---------------- producer ----------------
        int32_t b0[NC], bnd[NC];
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            b0[c] = 0;
            if (P.cols[c].dtype == TG_UTF8 && t_begin < t_end) b0[c] = __ldg(P.cols[c].offsets + t_begin * GT_ROWS);
        }
        uint32_t s = 0, ph = 0;
        for (int64_t tb = t_begin; tb < t_end; tb += 32) {
            // lane l: the end boundary of tile tb + l
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                bnd[c] = 0;
                if (P.cols[c].dtype == TG_UTF8) {
                    const int64_t r1 = min((tb + lane + 1) * (int64_t)GT_ROWS, P.n_rows);
                    bnd[c] = __ldg(P.cols[c].offsets + r1);
                }
            }
            const int n_here = (int)min((int64_t)32, t_end - tb);
            for (int i = 0; i < n_here; ++i) {
                const int64_t t = tb + i, r0 = t * GT_ROWS;
                const uint32_t rows = (uint32_t)min((int64_t)GT_ROWS, P.n_rows - r0);
                int32_t b1[NC];
#pragma unroll
                for (int c = 0; c < NC; ++c) b1[c] = __shfl_sync(0xffffffffu, bnd[c], i);
                if (lane == 0) {
                    mbar_wait(&empty[s], ph ^ 1u);
                    uint8_t* stage = ring + (size_t)s * P.stage_bytes;
                    const uint32_t vbytes = ((rows + 7) / 8 + 15) & ~15u;
                    uint32_t total = 0;
                    // sizes first (expect_tx precedes the copies)
                    uint32_t src_lo[NC], nbytes[NC];
#pragma unroll
                    for (int c = 0; c < NC; ++c) {
                        const GdCol& C = P.cols[c];
                        if (C.validity) total += vbytes;
                        src_lo[c] = 0;
                        nbytes[c] = 0;
                        if (C.dtype == TG_UTF8) {
                            total += ((rows + 1) * 4 + 15) & ~15u;
                            src_lo[c] = (uint32_t)b0[c] & ~15u;
                            nbytes[c] = (((uint32_t)b1[c] + 15u) & ~15u) - src_lo[c];
                            if (nbytes[c] > P.st[c].bytes_cap) nbytes[c] = 0;  // does not fit: consumers read global memory
                            s_byte_base[s][c] = nbytes[c] ? src_lo[c] : 0xFFFFFFFFu;
                            total += nbytes[c];
                        } else {
                            nbytes[c] = C.dtype == TG_BOOL ? vbytes : C.dtype == TG_INT32 || C.dtype == TG_FLOAT32 ? (rows * 4 + 15) & ~15u : (rows * 8 + 15) & ~15u;
                            total += nbytes[c];
                        }
                    }
                    for (int j = 0; j < P.n_jobs; ++j)
                        if ((P.tv_copy_mask >> j) & 1u) total += vbytes;
                    mbar_arrive_expect_tx(&full[s], total);
#pragma unroll
                    for (int c = 0; c < NC; ++c) {
                        const GdCol& C = P.cols[c];
                        if (C.validity) bulk_g2s(stage + P.st[c].val_off, reinterpret_cast<const uint8_t*>(C.validity) + r0 / 8, vbytes, &full[s]);
                        if (C.dtype == TG_UTF8) {
                            bulk_g2s(stage + P.st[c].main_off, C.offsets + r0, ((rows + 1) * 4 + 15) & ~15u, &full[s]);
                            if (nbytes[c]) bulk_g2s(stage + P.st[c].bytes_off, C.values + src_lo[c], nbytes[c], &full[s]);
                        } else {
                            const uint8_t* src = C.dtype == TG_BOOL ? C.values + r0 / 8
                                                 : C.dtype == TG_INT32 || C.dtype == TG_FLOAT32 ? C.values + r0 * 4 : C.values + r0 * 8;
                            bulk_g2s(stage + P.st[c].main_off, src, nbytes[c], &full[s]);
                        }
                    }
                    for (int j = 0; j < P.n_jobs; ++j)
                        if ((P.tv_copy_mask >> j) & 1u)
                            bulk_g2s(stage + P.st_target[j], reinterpret_cast<const uint8_t*>(P.jobs[j].target_validity) + r0 / 8, vbytes, &full[s]);
                }
#pragma unroll
                for (int c = 0; c < NC; ++c) b0[c] = b1[c];
                if (++s == P.n_stages) {
                    s = 0;
                    ph ^= 1u;
                }
            }
        }
    } else {
        // ---------------- consumers: one row per lane per tile ----------------
        // the counted groupings' descriptors live in registers (the loops over them are unrolled): table address, slots,
        // where the codes of their columns sit in `packed` (a two-column grouping reads its third code from bits 30..: 0)
        uint32_t j_tab[GD_MAX_JOBS], j_slots[GD_MAX_JOBS], j_shifts[GD_MAX_JOBS], j_tv[GD_MAX_JOBS];
        uint32_t* j_rows[GD_MAX_JOBS];
#pragma unroll
        for (int j = 0; j < GD_MAX_JOBS; ++j) {
            const GdJob& J = P.jobs[j];
            const bool counted = j < P.n_jobs && J.derived_from < 0;
            j_tab[j] = counted ? smem_u32(gd_smem + J.smem_off) : 0u;
            j_slots[j] = J.comp_slots;
            j_shifts[j] = (uint32_t)(10 * J.col[0]) | ((uint32_t)(10 * J.col[1]) << 8) | ((uint32_t)(J.n_cols > 2 ? 10 * J.col[2] : 30) << 16);
            j_tv[j] = P.st_target[j];
            j_rows[j] = J.cta_rows + (size_t)blockIdx.x * J.comp_slots;
        }
        uint32_t s = 0, ph = 0;
        const uint32_t rt0 = (uint32_t)warp * 32u + (uint32_t)lane;
        for (int64_t t = t_begin; t < t_end; ++t) {
            const int64_t r0 = t * GT_ROWS;
            const uint32_t rows = (uint32_t)min((int64_t)GT_ROWS, P.n_rows - r0);
            const uint32_t rt = min(rt0, rows - 1u);  // rows past the end: clamped for the loads, dropped at the counters
            const uint32_t row = (uint32_t)r0 + rt;
            mbar_wait(&full[s], ph);
            const uint8_t* stage = ring + (size_t)s * P.stage_bytes;
            uint32_t packed = 0;  // local code of column c in bits [10c ..) (NC <= 3)
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const GdCol& C = P.cols[c];
                const GdDict d = gd_dict(gd_smem, C.smem_off);
                uint32_t vbit = 1u;
                if (C.validity) vbit = (reinterpret_cast<const uint32_t*>(stage + P.st[c].val_off)[rt >> 5] >> (rt & 31u)) & 1u;
                uint64_t x, y = 0;
                uint32_t tag;
                if (C.dtype == TG_UTF8) {
                    const int32_t* so = reinterpret_cast<const int32_t*>(stage + P.st[c].main_off) + rt;
                    const int32_t b = so[0], len = so[1] - b;
                    const uint32_t base = s_byte_base[s][c];
                    if (base != 0xFFFFFFFFu) {
                        // the two aligned 8-byte words around the start, a 128-bit funnel shift, a length mask
                        const uint32_t pb = (uint32_t)b - base;
                        const uint2* vp = reinterpret_cast<const uint2*>(stage + P.st[c].bytes_off + (pb & ~7u));
                        const uint2 w0 = vp[0], w1 = vp[1];
                        const uint32_t sh = (pb & 7u) * 8u, sl = sh & 31u;
                        const bool up = sh >= 32u;
                        const uint32_t A = up ? w0.y : w0.x, Bw = up ? w1.x : w0.y, Cw = up ? w1.y : w1.x;
                        const uint32_t lo = __funnelshift_r(A, Bw, sl), hi = __funnelshift_r(Bw, Cw, sl);
                        const uint32_t nb = (uint32_t)min(len, 8) * 8u;  // bits kept
                        const uint32_t mlo = nb >= 32u ? 0xffffffffu : ((1u << nb) - 1u);
                        const uint32_t mhi = nb >= 64u ? 0xffffffffu : (nb > 32u ? ((1u << (nb - 32u)) - 1u) : 0u);
                        x = (uint64_t)(lo & mlo) | ((uint64_t)(hi & mhi) << 32);
                    } else {
                        x = len > 0 ? load_upto8(C.values, b, min(8, len)) : 0ull;
                    }
                    tag = (uint32_t)len + 1u;  // 1..9
                    if (len > 8 && vbit) {  // longer strings: identified by a 128-bit hash pair
                        const ulonglong2 h2 = gd_long_pair(C.values, b, b + len, x);
                        x = h2.x;
                        y = h2.y;
                        tag = GD_TAG_LONG;
                    }
                } else {
                    tag = 0x10u + (uint32_t)C.dtype;
                    const uint8_t* sv = stage + P.st[c].main_off;
                    switch (C.dtype) {
                        case TG_INT64: x = reinterpret_cast<const unsigned long long*>(sv)[rt]; break;
                        case TG_FLOAT64: x = canon_f64(reinterpret_cast<const unsigned long long*>(sv)[rt]); break;
                        case TG_INT32: x = (uint64_t)(int64_t) reinterpret_cast<const int32_t*>(sv)[rt]; break;
                        case TG_FLOAT32: x = canon_f64((uint64_t)__double_as_longlong((double)reinterpret_cast<const float*>(sv)[rt])); break;
                        default: x = (reinterpret_cast<const uint32_t*>(sv)[rt >> 5] >> (rt & 31u)) & 1u; break;  // TG_BOOL
                    }
                }
                if (!vbit) {
                    x = 0;
                    y = 0;
                    tag = GD_TAG_NULL;
                }
                int sl2 = (int)gd_hash(x, tag);
                bool hit = false;
#pragma unroll 1
                for (int probe = 0; probe < GD_PROBE; ++probe) {
                    const uint4 en = lds128_volatile(&d.ent[sl2]);
                    hit = en.z == tag && en.x == (uint32_t)x && en.y == (uint32_t)(x >> 32);
                    if (hit || en.z == 0u || en.z == GD_BUSY) break;
                    sl2 = (sl2 + 1) & (GD_DICT - 1);
                }
                if (!hit || tag == GD_TAG_LONG) sl2 = gd_lookup_slow(d, (uint32_t)sl2, x, y, tag, row);
                if (sl2 < 0) {
                    overflow = true;
                    sl2 = 0;
                }
                packed |= (uint32_t)sl2 << (10 * c);
            }
#pragma unroll
            for (int j = 0; j < GD_MAX_JOBS; ++j) {
                if (j_tab[j] == 0u) continue;  // absent or derived (warp-uniform)
                const uint32_t S = j_slots[j];
                uint32_t tbit = 1u;
                if (j_tv[j] != 0xFFFFFFFFu) tbit = (reinterpret_cast<const uint32_t*>(stage + j_tv[j])[rt >> 5] >> (rt & 31u)) & 1u;
                int cs = (int)((packed >> (j_shifts[j] & 255u)) & 1023u);
                uint32_t tot_a = j_tab[j], nul_a = j_tab[j] + GD_DICT * 4;  // shared-window addresses of the counters
                if (S) {
                    const uint32_t key = (uint32_t)cs | (((packed >> ((j_shifts[j] >> 8) & 255u)) & 1023u) << 10) |
                                         (((packed >> (j_shifts[j] >> 16)) & 1023u) << 20);
                    uint32_t h = key * 0x9E3779B1u;
                    h ^= h >> 15;
                    uint32_t sq = h & (S - 1);
                    bool hit = false;
#pragma unroll 1
                    for (int probe = 0; probe < GD_PROBE; ++probe) {
                        uint32_t v;
                        asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(j_tab[j] + sq * 4u));
                        hit = v == key;
                        if (hit || v == 0xFFFFFFFFu) break;
                        sq = (sq + 1) & (S - 1);
                    }
                    cs = hit ? (int)sq : gd_comp_slow(reinterpret_cast<uint32_t*>(gd_smem + P.jobs[j].smem_off), j_rows[j], S, sq, key, row, &s_comp_entries[j]);
                    if (cs < 0) overflow = true;
                    tot_a = j_tab[j] + S * 4u;
                    nul_a = j_tab[j] + S * 8u;
                }
                if (rt0 >= rows) cs = -1;  // a clamped row past the end
                // Few groups: one shared atomic per distinct counter per warp (plain per-lane shared atomics are 2x slower: the 32
                // lanes collide on a handful of counters). A composite table that already holds hundreds of groups spreads the lanes
                // over as many counters: two lanes rarely meet, and MATCH.ANY + the leader election cost more than the collisions.
                // (the lanes that took the slow path above may not have rejoined the others yet: the decision is read by one lane
                // after the warp has reconverged, so that every lane takes the same branch — the other one holds a full-mask MATCH)
                // — composite groupings only (S is warp-uniform): a single-column grouping pays nothing for the test)
                bool per_lane = false;
                if (S) {
                    __syncwarp();
                    uint32_t n_met = 0;
                    if (lane == 0) n_met = *reinterpret_cast<volatile uint32_t*>(&s_comp_entries[j]);
                    per_lane = __shfl_sync(0xffffffffu, n_met, 0) >= GT_DIRECT_GROUPS;
                }
                if (per_lane) {
                    if (cs >= 0) {
                        asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(tot_a + (uint32_t)cs * 4u), "r"(1u) : "memory");
                        if (!tbit) asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(nul_a + (uint32_t)cs * 4u), "r"(1u) : "memory");
                    }
                } else {
                    const unsigned peers = __match_any_sync(0xffffffffu, cs);
                    if (cs >= 0) {
                        if (lane == __ffs(peers) - 1)
                            asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(tot_a + (uint32_t)cs * 4u), "r"((uint32_t)__popc(peers)) : "memory");
                        if (!tbit) asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(nul_a + (uint32_t)cs * 4u), "r"(1u) : "memory");
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
            if (++s == P.n_stages) {
                s = 0;
                ph ^= 1u;
            }
        }
    }
    gd_fold<NC>(P, gd_smem, overflow, true);
}

// groups of a single-column grouping: the column's global dictionary slots; of a composite grouping: its key table
__global__ void gd_collect_kernel(const unsigned long long* present /* h1 or ckeys */, const unsigned long long* totals,
                                  const unsigned long long* nonnull, const long long* first_row, uint64_t cap, unsigned long long* out_n,
                                  uint64_t max_out, unsigned long long* out /* [max_out][3] = first_row, total, nonnull */) {
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += (uint64_t)gridDim.x * blockDim.x) {
        if (present[s] == EMPTY64) continue;
        const unsigned long long i = atomicAdd(out_n, 1ull);
        if (i < max_out) {
            out[i * 3 + 0] = (unsigned long long)first_row[s];
            out[i * 3 + 1] = totals[s];
            out[i * 3 + 2] = nonnull[s];
        }
    }
}

__global__ void group_collect_kernel(Table128 t, const unsigned long long* totals, const unsigned long long* nonnull,
                                     const long long* first_row, uint64_t cap, unsigned long long* out_n, uint64_t max_out,
                                     unsigned long long* out /* [max_out][3] = first_row, total, nonnull */) {
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += (uint64_t)gridDim.x * blockDim.x) {
        if (t.h1[s] == EMPTY64) continue;
        const unsigned long long i = atomicAdd(out_n, 1ull);
        if (i < max_out) {
            out[i * 3 + 0] = (unsigned long long)first_row[s];
            out[i * 3 + 1] = totals[s];
            out[i * 3 + 2] = nonnull[s];
        }
    }
}

// key values of the groups' first rows: per (group, column) -> {valid, start, length} (Utf8) or {valid, value bits, 0}
__global__ void group_keys_kernel(GrpParams P, const unsigned long long* groups /* [n][3] */, uint64_t n_groups,
                                  unsigned long long* meta /* [n][n_cols][3] */) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_groups * (uint64_t)P.n_cols) return;
    const uint64_t g = i / P.n_cols;
    const int c = (int)(i % P.n_cols);
    const int64_t row = (int64_t)groups[g * 3];
    const GrpCol& col = P.cols[c];
    unsigned long long valid = row_valid(col.validity, row) ? 1 : 0, x = 0, y = 0;
    if (valid) {
        switch (col.dtype) {
            case TG_UTF8: x = (unsigned long long)col.offsets[row]; y = (unsigned long long)(col.offsets[row + 1] - col.offsets[row]); break;
            case TG_INT64: case TG_FLOAT64: x = reinterpret_cast<const unsigned long long*>(col.values)[row]; break;
            case TG_INT32: x = (unsigned long long)(long long)reinterpret_cast<const int32_t*>(col.values)[row]; break;
            case TG_FLOAT32: x = (unsigned long long)__double_as_longlong((double)reinterpret_cast<const float*>(col.values)[row]); break;
            default: x = (reinterpret_cast<const uint32_t*>(col.values)[row >> 5] >> (row & 31)) & 1u; break;
        }
    }
    meta[i * 3 + 0] = valid;
    meta[i * 3 + 1] = x;
    meta[i * 3 + 2] = y;
}
// packs the Utf8 key bytes: one warp per (group, column) entry
__global__ void group_key_bytes_kernel(GrpParams P, const unsigned long long* meta, const unsigned long long* dst_off, uint64_t n_entries,
                                       uint8_t* dst) {
    const uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= n_entries) return;
    const GrpCol& col = P.cols[(int)(i % P.n_cols)];
    if (col.dtype != TG_UTF8 || !meta[i * 3]) return;
    const uint64_t src = meta[i * 3 + 1], len = meta[i * 3 + 2], d = dst_off[i];
    for (uint64_t k = lane; k < len; k += 32) dst[d + k] = col.values[src + k];
}

static size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static uint64_t pow2_at_least(uint64_t x) {
    uint64_t p = 1024;
    while (p < x) p <<= 1;
    return p;
}

struct GrpBatch {
    std::vector<int> aggs;                   // aggregate ids
    std::vector<Column*> dcols;              // distinct group columns
    std::vector<std::vector<int>> job_cols;  // per job: indices into dcols, in the grouping's order
};

// global tables of the dictionary path: a column's dictionary holds at most 148 CTAs x 1024 entries (and at most n)
static uint64_t gd_cap_dict(int64_t n) { return pow2_at_least(std::min<uint64_t>((uint64_t)n * 2, (uint64_t)1 << 18)); }
static uint64_t gd_cap_comp(int64_t n) { return pow2_at_least(std::min<uint64_t>((uint64_t)n * 2, (uint64_t)1 << 22)); }
static size_t grouped_dict_bytes(int64_t n, const GrpBatch& B) {
    size_t need = 256 + B.dcols.size() * gd_cap_dict(n) * 24;
    for (auto& jc : B.job_cols) need += jc.size() == 1 ? gd_cap_dict(n) * 16 : gd_cap_comp(n) * 32 + (size_t)GD_CTA_ROWS_BYTES;
    return need;
}

// fast path (column dictionaries): fills d_out[j] / n_groups[j]; returns false when the batch is not eligible or a CTA's
// shared tables overflowed (the caller then runs the generic kernel)
static bool grouped_count_dict(Engine& e, Table& t, Plan& p, const GrpBatch& B, uint8_t* scr, size_t out_b, std::vector<unsigned long long*>& d_out,
                               std::vector<unsigned long long>& n_groups) {
    const int64_t n = t.n_rows;
    const int nj = (int)B.aggs.size(), nc = (int)B.dcols.size();
    if (nc > GD_MAX_COLS || nj > GD_MAX_JOBS || n >= ((int64_t)1 << 31) || n <= 0) return false;
    int n_comp = 0;
    for (auto& jc : B.job_cols) {
        if (jc.size() > 3) return false;
        n_comp += jc.size() > 1;
    }
    if (getenv("TG_GROUPED_NO_DICT")) return false;
    GdParams P{};
    P.n_cols = nc;
    P.n_jobs = nj;
    P.n_rows = n;
    for (int j = 0; j < nj; ++j) {
        GdJob& J = P.jobs[j];
        J.target_validity = (const uint32_t*)t.find(p.aggs[B.aggs[j]].cols[0])->validity.p;
        J.n_cols = (int)B.job_cols[j].size();
        for (int k = 0; k < J.n_cols; ++k) J.col[k] = B.job_cols[j][k];
        J.derived_from = -1;
    }
    // marginals: a single-column grouping whose column is part of a composite grouping over the same target column is
    // summed out of that grouping's per-CTA table instead of being counted per row
    int n_derived = 0;
    for (int j = 0; j < nj; ++j) {
        if (P.jobs[j].n_cols != 1 || getenv("TG_GROUPED_NO_MARGINALS")) continue;
        for (int q2 = 0; q2 < nj && P.jobs[j].derived_from < 0; ++q2) {
            if (P.jobs[q2].n_cols < 2 || p.aggs[B.aggs[q2]].cols[0] != p.aggs[B.aggs[j]].cols[0]) continue;
            for (int k = 0; k < P.jobs[q2].n_cols; ++k)
                if (P.jobs[q2].col[k] == P.jobs[j].col[0]) {
                    P.jobs[j].derived_from = q2;
                    P.jobs[j].derived_pos = k;
                    ++n_derived;
                    break;
                }
        }
    }
    // ---- shared memory. Persistent part: dictionaries, counters of the counted single-column groupings, composite tables.
    const size_t budget = 222 * 1024;
    size_t stage_b = 0;
    uint32_t tv_off[GD_MAX_JOBS];
    {
        // one stage of the tile kernel's ring
        const size_t vb = round_up((size_t)(GT_ROWS + 7) / 8, 16);
        for (int c = 0; c < nc; ++c) {
            Column* col = B.dcols[c];
            GdStageCol& S = P.st[c];
            S.main_off = S.bytes_off = S.val_off = 0xFFFFFFFFu;
            S.bytes_cap = 0;
            if (col->validity.p) {
                S.val_off = (uint32_t)stage_b;
                stage_b += vb;
            }
            S.main_off = (uint32_t)stage_b;
            if (col->dtype == TG_UTF8) {
                stage_b += round_up((size_t)(GT_ROWS + 1) * 4, 16);
                // room for 1.5x the average tile plus slack (a tile with more bytes is read from global memory)
                const double avg = (double)col->value_bytes / (double)n;
                S.bytes_cap = (uint32_t)round_up((size_t)std::min(std::max(avg * GT_ROWS * 1.5 + 512.0, 2048.0), 24576.0), 16);
                S.bytes_off = (uint32_t)stage_b;
                stage_b += S.bytes_cap + 16;  // the funnel shift over-reads up to 16 bytes
            } else {
                stage_b += round_up((size_t)GT_ROWS * 8, 16);
            }
        }
        for (int j = 0; j < nj; ++j) {
            tv_off[j] = 0xFFFFFFFFu;
            if (!P.jobs[j].target_validity) continue;
            for (int q2 = 0; q2 < j; ++q2)
                if (P.jobs[q2].target_validity == P.jobs[j].target_validity) tv_off[j] = tv_off[q2];
            if (tv_off[j] == 0xFFFFFFFFu) {
                tv_off[j] = (uint32_t)stage_b;
                stage_b += vb;
            }
        }
    }
    bool tile = nc <= 3 && !getenv("TG_GROUPED_NO_TILE");
    uint32_t comp_slots = 0;
    size_t smem = 0;
    for (int attempt = 0; attempt < 2; ++attempt) {
        size_t off = 0;
        for (int c = 0; c < nc; ++c) {
            P.cols[c].smem_off = (uint32_t)off;
            off += GD_DICT_BYTES;
        }
        for (int j = 0; j < nj; ++j)
            if (P.jobs[j].n_cols == 1 && !(tile && P.jobs[j].derived_from >= 0)) {
                P.jobs[j].smem_off = (uint32_t)off;
                off += (size_t)GD_DICT * 8;
            }
        // the tile kernel keeps >= 2 stages of its ring (which also hosts the derived groupings' counters at the end)
        const size_t ring_min = tile ? std::max(3 * stage_b, (size_t)n_derived * GD_DICT * 8) : 0;
        if (off + ring_min > budget) {
            if (tile) {
                tile = false;
                continue;
            }
            return false;
        }
        comp_slots = 0;
        if (n_comp) {
            comp_slots = 8192;
            while (comp_slots > 2048 && off + ring_min + (size_t)comp_slots * 12 * (size_t)n_comp > budget) comp_slots >>= 1;
            if (off + ring_min + (size_t)comp_slots * 12 * (size_t)n_comp > budget) {
                if (tile) {
                    tile = false;
                    continue;
                }
                while (comp_slots > 256 && off + (size_t)comp_slots * 12 * (size_t)n_comp > budget) comp_slots >>= 1;
                if (off + (size_t)comp_slots * 12 * (size_t)n_comp > budget) return false;
            }
        }
        for (int j = 0; j < nj; ++j)
            if (P.jobs[j].n_cols > 1) {
                P.jobs[j].smem_off = (uint32_t)off;
                P.jobs[j].comp_slots = comp_slots;
                off += (size_t)comp_slots * 12;
            }
        if (tile) {
            P.ring_off = (uint32_t)off;
            P.stage_bytes = (uint32_t)stage_b;
            P.n_stages = (uint32_t)std::min<size_t>(GT_MAX_STAGES, (budget - off) / stage_b);
            size_t ring_b = (size_t)P.n_stages * stage_b, dq = 0;
            for (int j = 0; j < nj; ++j)
                if (P.jobs[j].n_cols == 1 && P.jobs[j].derived_from >= 0) {
                    P.jobs[j].smem_off = (uint32_t)(off + dq);
                    dq += (size_t)GD_DICT * 8;
                }
            ring_b = std::max(ring_b, dq);
            off += ring_b;
            for (int j = 0; j < nj; ++j) P.st_target[j] = tv_off[j];
            P.tv_copy_mask = 0;
            for (int j = 0; j < nj; ++j) {
                bool first = tv_off[j] != 0xFFFFFFFFu;
                for (int q2 = 0; q2 < j; ++q2) first = first && tv_off[q2] != tv_off[j];
                if (first) P.tv_copy_mask |= 1u << j;
            }
        }
        smem = off;
        break;
    }
    // global state (the caller sized the scratch block with grouped_dict_bytes)
    const uint64_t cap_d = gd_cap_dict(n), cap_c = gd_cap_comp(n);
    const size_t dcol_b = cap_d * 8 * 3, dsingle_b = cap_d * 8 * 2, dcomp_b = cap_c * 8 * 4;
    uint8_t* q = scr;
    unsigned int* d_over = (unsigned int*)q; q += 256;
    TG_CUDA(cudaMemsetAsync(d_over, 0, 256, e.stream));
    for (int c = 0; c < nc; ++c) {
        Column* col = B.dcols[c];
        GdCol& C = P.cols[c];
        C.values = col->values.p;
        C.offsets = (const int32_t*)col->offsets.p;
        C.validity = (const uint32_t*)col->validity.p;
        C.dtype = col->dtype;
        C.dict = Table128{(unsigned long long*)q, (unsigned long long*)(q + cap_d * 8), nullptr, cap_d - 1};
        C.first_row = (long long*)(q + cap_d * 16);
        TG_CUDA(cudaMemsetAsync(q, 0xFF, cap_d * 16, e.stream));
        TG_CUDA(cudaMemsetAsync(q + cap_d * 16, 0x7F, cap_d * 8, e.stream));
        q += dcol_b;
    }
    for (int j = 0; j < nj; ++j) {
        GdJob& J = P.jobs[j];
        if (J.n_cols == 1) {
            J.totals = (unsigned long long*)q;
            J.nonnull = (unsigned long long*)(q + cap_d * 8);
            TG_CUDA(cudaMemsetAsync(q, 0, cap_d * 16, e.stream));
            q += dsingle_b;
        } else {
            J.ckeys = (unsigned long long*)q;
            J.totals = (unsigned long long*)(q + cap_c * 8);
            J.nonnull = (unsigned long long*)(q + cap_c * 16);
            J.crow = (long long*)(q + cap_c * 24);
            J.cta_rows = (uint32_t*)(q + dcomp_b);
            J.cmask = cap_c - 1;
            TG_CUDA(cudaMemsetAsync(q, 0xFF, cap_c * 8, e.stream));
            TG_CUDA(cudaMemsetAsync(q + cap_c * 8, 0, cap_c * 16, e.stream));
            TG_CUDA(cudaMemsetAsync(q + cap_c * 24, 0x7F, cap_c * 8, e.stream));
            q += dcomp_b + GD_CTA_ROWS_BYTES;
        }
    }
    P.overflow = d_over;
    typedef void (*Kern)(const GdParams);
    if (tile) {
        const Kern kern = nc == 1 ? (Kern)group_count_tile_kernel<1> : nc == 2 ? (Kern)group_count_tile_kernel<2> : (Kern)group_count_tile_kernel<3>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  // per device
        const int64_t n_tiles = (n + GT_ROWS - 1) / GT_ROWS;
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(n_tiles, (int64_t)e.sm_count));
        kern<<<grid, GT_THREADS, smem, e.stream>>>(P);
    } else {
        const Kern kern = nc == 1 ? (Kern)group_count_dict_kernel<1> : nc == 2 ? (Kern)group_count_dict_kernel<2>
                          : nc == 3 ? (Kern)group_count_dict_kernel<3> : (Kern)group_count_dict_kernel<4>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  // per device
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((n + GD_THREADS * GD_ILP - 1) / (GD_THREADS * GD_ILP), (int64_t)e.sm_count));
        kern<<<grid, GD_THREADS, smem, e.stream>>>(P);
    }
    TG_CUDA(cudaGetLastError());
    // the overflow flag is read together with the group counts (ONE synchronisation): the collection kernels are cheap
    // enough to run speculatively
    // the groups: out triples behind the tables (the generic path's out area is not used by this path)
    unsigned long long* d_cnt = (unsigned long long*)(d_over + 16);
    const int cgrid = (int)std::max<uint64_t>(1, std::min<uint64_t>((std::max(cap_d, cap_c) + 255) / 256, (uint64_t)e.sm_count * 8));
    for (int j = 0; j < nj; ++j) {
        const GdJob& J = P.jobs[j];
        if (J.n_cols == 1) {
            const GdCol& C = P.cols[J.col[0]];
            gd_collect_kernel<<<cgrid, 256, 0, e.stream>>>(C.dict.h1, J.totals, J.nonnull, C.first_row, cap_d, d_cnt + j, GRP_MAX_GROUPS_DEV, d_out[j]);
        } else {
            gd_collect_kernel<<<cgrid, 256, 0, e.stream>>>(J.ckeys, J.totals, J.nonnull, J.crow, cap_c, d_cnt + j, GRP_MAX_GROUPS_DEV, d_out[j]);
        }
        TG_CUDA(cudaGetLastError());
    }
    // d_over (4 bytes) and d_cnt (64 bytes behind it) come back in one pinned copy
    unsigned long long* h_cnt = (unsigned long long*)e.host_scratch(256);
    TG_CUDA(cudaMemcpyAsync(h_cnt, d_over, 64 + GD_MAX_JOBS * 8, cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    p.stats.launches += 1 + nj;
    e.launches += 1 + nj;
    if (*(const unsigned int*)h_cnt) return false;
    for (int j = 0; j < nj; ++j) n_groups[j] = h_cnt[8 + j];
    (void)out_b;
    return true;
}

// generic path (128-bit fingerprints, any number of columns / groups)
static void grouped_count_generic(Engine& e, Table& t, Plan& p, const GrpBatch& B, uint8_t* scr, size_t per_job, uint64_t cap,
                                  std::vector<unsigned long long*>& d_out, std::vector<unsigned long long>& n_groups) {
    const int64_t n = t.n_rows;
    const int nj = (int)B.aggs.size();
    const size_t h_b = cap * 8;
    GrpParams P{};
    P.n_cols = (int)B.dcols.size();
    P.n_jobs = nj;
    P.n_rows = n;
    for (size_t i = 0; i < B.dcols.size(); ++i)
        P.cols[i] = GrpCol{B.dcols[i]->values.p, (const int32_t*)B.dcols[i]->offsets.p, (const uint32_t*)B.dcols[i]->validity.p, B.dcols[i]->dtype, 0u, 0u, 0u};
    std::vector<unsigned long long*> d_n(nj);
    for (int j = 0; j < nj; ++j) {
        uint8_t* q = scr + (size_t)j * per_job;
        GrpJob& J = P.jobs[j];
        J.gt = Table128{(unsigned long long*)q, (unsigned long long*)(q + h_b), nullptr, cap - 1}; q += 2 * h_b;
        J.totals = (unsigned long long*)q; q += h_b;
        J.nonnull = (unsigned long long*)q; q += h_b;
        J.first_row = (long long*)q; q += h_b;
        d_n[j] = (unsigned long long*)q;
        J.n_groups = d_n[j];
        J.target_validity = (const uint32_t*)t.find(p.aggs[B.aggs[j]].cols[0])->validity.p;
        // the fingerprint folds a grouping's columns in the batch's column order; "first" = the lowest index it contains
        int lowest = GRP_MAX_COLS;
        for (int ci : B.job_cols[j]) {
            P.cols[ci].job_mask |= 1u << j;
            lowest = std::min(lowest, ci);
        }
        P.cols[lowest].first_mask |= 1u << j;
        TG_CUDA(cudaMemsetAsync(J.gt.h1, 0xFF, 2 * h_b, e.stream));
        TG_CUDA(cudaMemsetAsync(J.totals, 0, 2 * h_b, e.stream));
        TG_CUDA(cudaMemsetAsync(J.first_row, 0x7F, h_b, e.stream));
        TG_CUDA(cudaMemsetAsync(d_n[j], 0, 256, e.stream));
    }
    // shared tables: a multi-column grouping has (up to) the product of its columns' cardinalities as groups, so it gets
    // sixteen shares of the block where a single-column grouping gets one; every table a power of two, at most 8192 slots
    int shares = 0;
    for (int j = 0; j < nj; ++j) shares += B.job_cols[j].size() > 1 ? 16 : 1;
    size_t smem_slots = 0;
    for (int j = 0; j < nj; ++j) {
        const size_t want = (size_t)GRP_SMEM_BYTES / 24 * (B.job_cols[j].size() > 1 ? 16 : 1) / (size_t)shares;
        int sl = 512;
        while ((size_t)sl * 2 <= want && sl < 8192) sl <<= 1;
        P.slots[j] = sl;
        P.slot_base[j] = (int32_t)smem_slots;
        smem_slots += (size_t)sl;
    }
    const size_t smem = smem_slots * 24;
    typedef void (*Kern)(const GrpParams);
    const Kern kern = nj == 1 ? (Kern)group_count_fused_kernel<1> : nj == 2 ? (Kern)group_count_fused_kernel<2>
                      : nj == 3 ? (Kern)group_count_fused_kernel<3> : (Kern)group_count_fused_kernel<4>;
    TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  // per device
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((n + GRP_THREADS * GRP_ILP - 1) / (GRP_THREADS * GRP_ILP), (int64_t)e.sm_count));
    kern<<<grid, GRP_THREADS, smem, e.stream>>>(P);
    TG_CUDA(cudaGetLastError());
    const int cgrid = (int)std::max<uint64_t>(1, std::min<uint64_t>((cap + 255) / 256, (uint64_t)e.sm_count * 8));
    std::vector<unsigned long long> h_n((size_t)nj * 2, 0);
    for (int j = 0; j < nj; ++j) {
        const GrpJob& J = P.jobs[j];
        group_collect_kernel<<<cgrid, 256, 0, e.stream>>>(J.gt, J.totals, J.nonnull, J.first_row, cap, d_n[j] + 1, GRP_MAX_GROUPS_DEV, d_out[j]);
        TG_CUDA(cudaGetLastError());
        TG_CUDA(cudaMemcpyAsync(&h_n[(size_t)j * 2], d_n[j], 16, cudaMemcpyDeviceToHost, e.stream));
    }
    TG_CUDA(cudaStreamSynchronize(e.stream));
    p.stats.launches += 1 + nj;
    e.launches += 1 + nj;
    for (int j = 0; j < nj; ++j) n_groups[j] = h_n[(size_t)j * 2];
}

// One batch = up to GRP_MAX_JOBS groupings over up to GRP_MAX_COLS distinct group columns: one launch of a counting kernel
// (column dictionaries when the batch is narrow and its groups are few, 128-bit fingerprints otherwise), then per
// grouping the collection of the groups and of their key values.
static void run_grouped_batch(Engine& e, Table& t, Plan& p, const GrpBatch& B) {
    const std::vector<int>& batch = B.aggs;
    const std::vector<Column*>& dcols = B.dcols;
    const std::vector<std::vector<int>>& job_cols = B.job_cols;
    const int64_t n = t.n_rows;
    const int nj = (int)batch.size();
    // algorithmic bytes: every distinct group column once, every distinct target bitmap once
    for (auto* c : dcols) {
        uint64_t b = c->validity.p ? (uint64_t)(n + 7) / 8 : 0;
        if (c->dtype == TG_UTF8) b += (uint64_t)(n + 1) * 4 + (uint64_t)c->value_bytes;
        else if (c->dtype == TG_BOOL) b += (uint64_t)(n + 7) / 8;
        else b += (uint64_t)n * c->elem_bytes();
        p.stats.bytes_scanned += b;
    }
    {
        std::vector<const uint8_t*> seen;
        for (int id : batch) {
            Column* target = t.find(p.aggs[id].cols[0]);
            if (target->validity.p && std::find(seen.begin(), seen.end(), target->validity.p) == seen.end()) {
                seen.push_back(target->validity.p);
                p.stats.bytes_scanned += (uint64_t)(n + 7) / 8;
            }
        }
    }
    if (n == 0) {  // an empty shard: no groups
        for (int id : batch) {
            p.aggs[id].blob.assign(8, 0);
        }
        return;
    }
    const uint64_t cap = pow2_at_least(std::min<uint64_t>((uint64_t)n * 2, GRP_MAX_GROUPS_DEV * 4));
    const size_t h_b = cap * 8, out_b = round_up((size_t)GRP_MAX_GROUPS_DEV * 24, 256);
    const size_t per_job = 5 * h_b + 512;
    // [tables of the counting kernel (either path)][out triples: nj x out_b]
    const size_t tables_b = round_up(std::max(per_job * (size_t)nj, grouped_dict_bytes(n, B)), 256);
    uint8_t* scr = e.scratch(tables_b + out_b * (size_t)nj + 1024);
    std::vector<unsigned long long*> d_out(nj);
    std::vector<unsigned long long> n_groups_v((size_t)nj, 0);
    for (int j = 0; j < nj; ++j) d_out[j] = (unsigned long long*)(scr + tables_b + out_b * (size_t)j);
    cudaEventRecord(e.ev[4], e.stream);
    if (!grouped_count_dict(e, t, p, B, scr, out_b, d_out, n_groups_v)) grouped_count_generic(e, t, p, B, scr, per_job, cap, d_out, n_groups_v);
    cudaEventRecord(e.ev[5], e.stream);
    TG_CUDA(cudaStreamSynchronize(e.stream));
    float ms = 0;
    cudaEventElapsedTime(&ms, e.ev[4], e.ev[5]);
    p.stats.hash_ms += ms;
    p.stats.gpu_ms += ms;

    // ---- key values of the groups, all groupings of the batch together: three waves of small kernels / copies through
    // pinned memory and ONE synchronisation per wave, however many groupings and groups there are ----
    struct Fetch {
        std::vector<Column*> gcols;
        GrpParams PK{};
        size_t nc = 0, n_entries = 0;
        unsigned long long ng = 0;
        bool live = false;
        std::vector<unsigned long long> out, meta, dst_off;
        std::vector<uint8_t> key_bytes;
        unsigned long long *d_meta = nullptr, *d_dst = nullptr;
        uint8_t* d_bytes = nullptr;
        bool own_bytes = false;
        uint64_t total = 0;
        size_t h_off = 0;
    };
    std::vector<Fetch> F((size_t)nj);
    size_t aux_b = 0, host_b = 0;
    for (int j = 0; j < nj; ++j) {
        Fetch& f = F[j];
        Agg& a = p.aggs[batch[j]];
        f.ng = n_groups_v[j];
        if (f.ng > GRP_MAX_GROUPS_DEV) {
            a.err = TG_ERR_UNSUPPORTED;
            a.err_msg = "grouped completeness: more than 1048576 groups";
            continue;
        }
        f.live = true;
        for (int ci : job_cols[j]) f.gcols.push_back(dcols[ci]);
        f.PK.n_cols = (int)f.gcols.size();  // the key kernels see the grouping's own columns, in its own order
        f.PK.n_rows = n;
        for (size_t i = 0; i < f.gcols.size(); ++i)
            f.PK.cols[i] = GrpCol{f.gcols[i]->values.p, (const int32_t*)f.gcols[i]->offsets.p, (const uint32_t*)f.gcols[i]->validity.p, f.gcols[i]->dtype, 0u, 0u, 0u};
        f.nc = f.gcols.size();
        f.n_entries = (size_t)f.ng * f.nc;
        f.h_off = host_b;
        host_b += round_up((size_t)f.ng * 24 + f.n_entries * 24, 256);
        aux_b += round_up(f.n_entries * 32, 256);
    }
    // wave 1: group triples + key metadata
    if (host_b) {
        uint8_t* d_auxp = e.aux(aux_b + 256);  // grow-only auxiliary block (no cudaMalloc per execute)
        uint8_t* h = e.host_scratch(host_b);
        for (int j = 0; j < nj; ++j) {
            Fetch& f = F[j];
            if (!f.live || !f.ng) continue;
            f.d_meta = (unsigned long long*)d_auxp;
            f.d_dst = f.d_meta + f.n_entries * 3;
            d_auxp += round_up(f.n_entries * 32, 256);
            TG_CUDA(cudaMemcpyAsync(h + f.h_off, d_out[j], (size_t)f.ng * 24, cudaMemcpyDeviceToHost, e.stream));
            group_keys_kernel<<<(unsigned)((f.n_entries + 255) / 256), 256, 0, e.stream>>>(f.PK, d_out[j], f.ng, f.d_meta);
            TG_CUDA(cudaGetLastError());
            TG_CUDA(cudaMemcpyAsync(h + f.h_off + (size_t)f.ng * 24, f.d_meta, f.n_entries * 24, cudaMemcpyDeviceToHost, e.stream));
            p.stats.launches += 1;
            e.launches += 1;
        }
        TG_CUDA(cudaStreamSynchronize(e.stream));
        for (int j = 0; j < nj; ++j) {
            Fetch& f = F[j];
            if (!f.live || !f.ng) continue;
            const unsigned long long* ho = (const unsigned long long*)(h + f.h_off);
            f.out.assign(ho, ho + (size_t)f.ng * 3);
            f.meta.assign(ho + (size_t)f.ng * 3, ho + (size_t)f.ng * 3 + f.n_entries * 3);
            f.dst_off.assign(f.n_entries, 0);
            for (size_t i = 0; i < f.n_entries; ++i) {
                f.dst_off[i] = f.total;
                if (f.gcols[i % f.nc]->dtype == TG_UTF8 && f.meta[i * 3]) f.total += f.meta[i * 3 + 2];
            }
        }
        // wave 2: the Utf8 key bytes, packed per grouping where its triples were (the scratch block, >= max_groups * 24 bytes)
        size_t hb = 0;
        for (int j = 0; j < nj; ++j) {
            Fetch& f = F[j];
            if (f.total) {
                f.h_off = hb;
                hb += round_up(f.n_entries * 8, 256) + round_up((size_t)f.total, 256);
            }
        }
        if (hb) {
            h = e.host_scratch(hb);
            cudaError_t ce = cudaSuccess;
            for (int j = 0; j < nj && ce == cudaSuccess; ++j) {
                Fetch& f = F[j];
                if (!f.total) continue;
                f.d_bytes = f.total <= out_b ? (uint8_t*)d_out[j] : nullptr;
                f.own_bytes = f.d_bytes == nullptr;
                if (f.own_bytes) ce = cudaMalloc(&f.d_bytes, (size_t)f.total);
                if (ce != cudaSuccess) break;
                memcpy(h + f.h_off, f.dst_off.data(), f.n_entries * 8);
                ce = cudaMemcpyAsync(f.d_dst, h + f.h_off, f.n_entries * 8, cudaMemcpyHostToDevice, e.stream);
                if (ce != cudaSuccess) break;
                group_key_bytes_kernel<<<(unsigned)((f.n_entries * 32 + 255) / 256), 256, 0, e.stream>>>(f.PK, f.d_meta, f.d_dst, f.n_entries, f.d_bytes);
                ce = cudaGetLastError();
                if (ce == cudaSuccess)
                    ce = cudaMemcpyAsync(h + f.h_off + round_up(f.n_entries * 8, 256), f.d_bytes, (size_t)f.total, cudaMemcpyDeviceToHost, e.stream);
                p.stats.launches += 1;
                e.launches += 1;
            }
            const cudaError_t se = cudaStreamSynchronize(e.stream);
            if (ce == cudaSuccess) ce = se;
            for (auto& f : F)
                if (f.own_bytes && f.d_bytes) cudaFree(f.d_bytes);
            TG_CUDA(ce);
            for (auto& f : F)
                if (f.total) f.key_bytes.assign(h + f.h_off + round_up(f.n_entries * 8, 256), h + f.h_off + round_up(f.n_entries * 8, 256) + f.total);
        }
    }
    for (int j = 0; j < nj; ++j) {
        Fetch& f = F[j];
        if (!f.live) continue;
        Agg& a = p.aggs[batch[j]];
        const unsigned long long n_groups = f.ng;
        const size_t nc = f.nc;
        // blob: [u64 n_groups] then per group: u32 key_len, key (group column values joined by \x1f), u64 total, u64 non_null
        a.blob.resize(8);
        memcpy(a.blob.data(), &n_groups, 8);
        std::string key;
        for (unsigned long long g = 0; g < n_groups; ++g) {
            key.clear();
            for (size_t i = 0; i < nc; ++i) {
                if (i) key += '\x1f';
                const size_t en = (size_t)g * nc + i;
                if (!f.meta[en * 3]) {
                    // (a value histogram must tell the NULL group from the string 'NULL' when shard states are merged by key:
                    // its NULL key starts with a byte no valid UTF-8 value holds)
                    key += (a.flags & 2) ? "\xFFNULL" : "NULL";
                    continue;
                }
                const unsigned long long x = f.meta[en * 3 + 1];
                switch (f.gcols[i]->dtype) {
                    case TG_UTF8: key.append((const char*)f.key_bytes.data() + f.dst_off[en], (size_t)f.meta[en * 3 + 2]); break;
                    case TG_INT64: case TG_INT32: key += fmt_i64((int64_t)x); break;
                    case TG_FLOAT64: case TG_FLOAT32: {
                        double d;
                        memcpy(&d, &x, 8);
                        key += fmt_f64(d);
                    } break;
                    default:  // Boolean group values print as the empty string, as before (unpinned, DESIGN §5); a value histogram casts them to VARCHAR
                        if (a.flags & 2) key += x ? "true" : "false";
                        break;
                }
            }
            uint32_t L = (uint32_t)key.size();
            size_t o = a.blob.size();
            a.blob.resize(o + 4 + L + 16);
            memcpy(a.blob.data() + o, &L, 4);
            memcpy(a.blob.data() + o + 4, key.data(), L);
            memcpy(a.blob.data() + o + 4 + L, &f.out[g * 3 + 1], 8);
            memcpy(a.blob.data() + o + 4 + L + 8, &f.out[g * 3 + 2], 8);
        }
    }
}

// All grouped-completeness aggregates of a plan: bound to their columns, packed into batches that share one pass
void exec_grouped_jobs(Engine& e, Table& t, Plan& p, const std::vector<int>& agg_ids) {
    std::vector<int> batch;
    std::vector<Column*> dcols;
    std::vector<std::vector<int>> job_cols;
    auto flush = [&]() {
        if (!batch.empty()) run_grouped_batch(e, t, p, GrpBatch{batch, dcols, job_cols});
        batch.clear();
        dcols.clear();
        job_cols.clear();
    };
    for (int id : agg_ids) {
        Agg& a = p.aggs[id];
        try {
            auto need_col = [&](const std::string& name) -> Column* {
                Column* c = t.find(name);
                if (!c) throw Error(TG_ERR_COLUMN_NOT_FOUND, "Schema error: No field named " + name + ". Valid fields are " + t.valid_fields() + ".");
                return c;
            };
            need_col(a.cols[0]);
            std::vector<Column*> gcols;
            for (size_t i = 1; i < a.cols.size(); ++i) gcols.push_back(need_col(a.cols[i]));
            if (gcols.size() > (size_t)GRP_MAX_COLS) throw Error(TG_ERR_UNSUPPORTED, "grouped completeness: more than 8 grouping columns");
            if ((a.flags & 2) && (gcols[0]->dtype == TG_FLOAT64 || gcols[0]->dtype == TG_FLOAT32 || gcols[0]->temporal))
                throw Error(TG_ERR_UNSUPPORTED, "histogram of a floating-point / temporal column: CAST(" + a.cols[1] + " AS VARCHAR) formatting is not restated");
            uint64_t zero = 0;
            a.blob.assign((uint8_t*)&zero, (uint8_t*)&zero + 8);
            if (t.n_rows == 0) continue;
            // does it fit the open batch?
            std::vector<Column*> merged = dcols;
            for (auto* c : gcols)
                if (std::find(merged.begin(), merged.end(), c) == merged.end()) merged.push_back(c);
            if (batch.size() == (size_t)GRP_MAX_JOBS || merged.size() > (size_t)GRP_MAX_COLS) {
                flush();
                merged.clear();
                for (auto* c : gcols)
                    if (std::find(merged.begin(), merged.end(), c) == merged.end()) merged.push_back(c);
            }
            dcols = merged;
            std::vector<int> idx;
            for (auto* c : gcols) idx.push_back((int)(std::find(dcols.begin(), dcols.end(), c) - dcols.begin()));
            batch.push_back(id);
            job_cols.push_back(idx);
        } catch (Error& er) {
            if (er.code == TG_ERR_CUDA) throw;
            a.err = er.code;
            a.err_msg = er.msg;
        }
    }
    flush();
}

}  // namespace tg
