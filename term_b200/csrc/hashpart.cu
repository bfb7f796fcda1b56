// K3 (large inputs) — radix-partitioned hash jobs over a single Int64 / Float64 key column.
//
// Replaces  COUNT(DISTINCT c) / GROUP BY c HAVING COUNT(*) = 1                   constraints/uniqueness.rs:549-718
//           LEFT JOIN .. WHERE parent IS NULL -> COUNT(*), COUNT(DISTINCT child)  constraints/foreign_key.rs:165-172
// for key columns too large for an L2-resident hash table.
//
// Measured on B200 (tools/micro/atomics_bench.cu): random 64-bit atomicCAS runs at ~110 G/s while the table fits
// in L2 (<= 64 MB) and at ~21 G/s once it lives in HBM; random loads 280 G/s vs 40 G/s. So instead of one 2n-slot
// table in HBM the keys are first radix-partitioned by hash bits 32.. into P buckets of <= ~3 M keys (two
// streaming passes: histogram, then a scatter that reorders each 2048-key tile in shared memory so every bucket
// run leaves the SM as one coalesced burst), and the buckets are then deduplicated one after another in ONE reused,
// L2-resident 64 MB table (keys only; "seen twice" is a 1-bit-per-slot bitmap, so the second atomic only happens
// for duplicates). The same histogram/scatter pair with the rank field of the hash is step 1 of the multi-GPU
// all-to-all shuffle.
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "hash_common.cuh"
#include "hashpart.hpp"

namespace tg {

constexpr int PART_THREADS = 256;
constexpr int PART_KEYS_PER_THREAD = 8;
constexpr int PART_TILE = PART_THREADS * PART_KEYS_PER_THREAD;  // 2048 keys per CTA iteration
constexpr int PART_MAX = 1024;                                   // buckets
constexpr int64_t BUCKET_TARGET_KEYS = 2ll << 20;                // keys per bucket -> 8M-slot (64 MB) table, load <= 0.25

// tunables (environment overrides are for the sweep in tools/; the defaults are the measured optimum on B200)
static int64_t bucket_target_keys() {
    static const int64_t v = [] {
        const char* e = getenv("TG_HASH_BUCKET_KEYS");
        const long long x = e ? atoll(e) : 0;
        return x > 1024 ? (int64_t)x : BUCKET_TARGET_KEYS;
    }();
    return v;
}
static uint64_t slots_factor() {
    static const uint64_t v = [] {
        const char* e = getenv("TG_HASH_SLOTS_FACTOR");
        const long long x = e ? atoll(e) : 0;
        return x >= 2 ? (uint64_t)x : (uint64_t)4;
    }();
    return v;
}
size_t distinct64_min_rows() { return (size_t)bucket_target_keys(); }

struct PartCounters {
    unsigned long long nulls;
    unsigned long long special;  // rows whose key equals the EMPTY sentinel (kept out of the tables)
    unsigned long long pad[2];
};

// MODE 0: local radix bucket (hash bits 32..), EMPTY-sentinel keys and NULLs are counted and skipped
// MODE 1: destination rank of the shuffle, every valid key is kept (raw bits)
// MODE 2: destination rank by VALUE RANGE (Int64 keys known to be dense): part = (key - range_min) / range_span, so every
//         rank receives a contiguous slice of the key space and de-duplicates it with the bitmap path
// MODE 3: destination rank by SPLITTERS (the distributed sort of K6): part = number of splitters < key, so part p holds
//         the keys in (splitter[p-1], splitter[p]] and equal keys meet on one rank; an optional payload travels along
enum { PM_BUCKET = 0, PM_RANK = 1, PM_RANGE = 2, PM_SPLIT = 3 };
struct RangeSplit {
    long long min;
    unsigned long long span;
    const uint64_t* splitters = nullptr;  // PM_SPLIT: parts - 1 ascending keys (device)
    // PM_RANGE: part = mulhi(key - min, inv), inv = min(2^64 - 1, ceil(2^64 / span)) — monotone in the key and within one
    // of the exact quotient, which is all a partition needs (a 64-bit division per key tripled the histogram pass)
    unsigned long long inv = 0;
    static RangeSplit range(long long mn, unsigned long long span) {
        RangeSplit r{mn, span};
        r.inv = span <= 1 ? ~0ull : (unsigned long long)((((unsigned __int128)1 << 64) + span - 1) / span);
        return r;
    }
};

// Loads the PART_KEYS_PER_THREAD keys of this thread's tile slots up front (independent, predicated loads: all in
// flight together) and classifies them from registers: part >= 0, -1 NULL / past the end, -2 the EMPTY sentinel
// (MODE 0 only; it is counted and kept out of the tables).
template <int MODE>
__device__ __forceinline__ void load_classify(const uint64_t* __restrict__ values, const uint32_t* __restrict__ validity, int64_t base,
                                              int64_t n, int is_f64, uint32_t parts, uint64_t (&key)[PART_KEYS_PER_THREAD],
                                              int (&part)[PART_KEYS_PER_THREAD], RangeSplit rs = RangeSplit{0, 1}) {
    uint64_t raw[PART_KEYS_PER_THREAD];
    uint32_t vw[PART_KEYS_PER_THREAD];
#pragma unroll
    for (int k = 0; k < PART_KEYS_PER_THREAD; ++k) {
        const int64_t row = base + k * PART_THREADS + threadIdx.x;
        const bool in = row < n;
        raw[k] = in ? __ldg(values + row) : 0ull;
        vw[k] = in ? (validity ? __ldg(validity + (row >> 5)) : 0xffffffffu) : 0u;
    }
#pragma unroll
    for (int k = 0; k < PART_KEYS_PER_THREAD; ++k) {
        const int64_t row = base + k * PART_THREADS + threadIdx.x;
        const bool valid = (vw[k] >> (row & 31)) & 1u;
        const uint64_t ck = is_f64 ? canon_f64(raw[k]) : raw[k];
        const uint64_t h = fmix64(ck);
        if (MODE == PM_BUCKET) {
            key[k] = ck;
            part[k] = !valid ? -1 : (ck == EMPTY64 ? -2 : (int)hash_bucket(h, parts - 1));
        } else if (MODE == PM_RANK) {
            key[k] = raw[k];
            part[k] = !valid ? -1 : (int)hash_rank(h, parts);
        } else if (MODE == PM_RANGE) {
            key[k] = raw[k];
            const unsigned long long d = (long long)raw[k] < rs.min ? 0ull  // (below a sampled minimum: the first part)
                                                                    : __umul64hi((unsigned long long)raw[k] - (unsigned long long)rs.min, rs.inv);
            part[k] = !valid ? -1 : (int)(d < parts ? d : parts - 1);
        } else {
            key[k] = raw[k];
            int lo = 0, hi = (int)parts - 1;  // first splitter >= key (lower bound) = number of splitters < key
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (__ldg(rs.splitters + mid) < raw[k]) lo = mid + 1;
                else hi = mid;
            }
            part[k] = !valid ? -1 : lo;
        }
    }
}

template <int MODE>
__global__ void __launch_bounds__(PART_THREADS) part_hist_kernel(const uint64_t* __restrict__ values, const uint32_t* __restrict__ validity,
                                                                 int64_t n, int is_f64, uint32_t parts, unsigned long long* hist,
                                                                 PartCounters* ctr, RangeSplit rs = RangeSplit{0, 1}) {
    // `copies` private histograms (one per group of warps) keep same-address shared atomics rare for small `parts`
    __shared__ uint32_t s_hist[PART_MAX];
    const uint32_t copies = parts <= PART_MAX / 8 ? 8u : 1u;
    for (int i = threadIdx.x; i < (int)(parts * copies); i += PART_THREADS) s_hist[i] = 0;
    __syncthreads();
    uint32_t* my_hist = s_hist + ((threadIdx.x >> 5) % copies) * parts;
    unsigned long long nulls = 0, special = 0;
    const int64_t n_tiles = (n + PART_TILE - 1) / PART_TILE;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t base = tile * PART_TILE;
        uint64_t key[PART_KEYS_PER_THREAD];
        int part[PART_KEYS_PER_THREAD];
        load_classify<MODE>(values, validity, base, n, is_f64, parts, key, part, rs);
        // (Measured and dropped here — unlike in the scatter, whose atomics RETURN a value: aggregating equal parts across the
        // warp first, 0.41 vs 0.35 ms per GB of keys; two tiles per iteration for more loads in flight, 0.62 ms.)
#pragma unroll
        for (int k = 0; k < PART_KEYS_PER_THREAD; ++k) {
            if (part[k] >= 0) atomicAdd(&my_hist[part[k]], 1u);
            if (part[k] == -2) ++special;
            else if (part[k] == -1 && base + k * PART_THREADS + threadIdx.x < n) ++nulls;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < (int)parts; i += PART_THREADS) {
        uint32_t v = 0;
        for (uint32_t c = 0; c < copies; ++c) v += s_hist[c * parts + i];
        if (v) atomicAdd(&hist[i], (unsigned long long)v);
    }
    flush_counter(nulls, &ctr->nulls);
    flush_counter(special, &ctr->special);
}

// exclusive prefix of the histogram -> offsets[parts + 1]; cursors[parts] = offsets (consumed by the scatter)
__global__ void part_prefix_kernel(const unsigned long long* hist, uint32_t parts, unsigned long long* offsets, unsigned long long* cursors) {
    __shared__ unsigned long long s[PART_MAX];
    const int t = threadIdx.x;
    s[t] = t < (int)parts ? hist[t] : 0;
    __syncthreads();
    for (int d = 1; d < PART_MAX; d <<= 1) {
        const unsigned long long v = t >= d ? s[t - d] : 0;
        __syncthreads();
        s[t] += v;
        __syncthreads();
    }
    if (t < (int)parts) {
        const unsigned long long ex = t ? s[t - 1] : 0;
        offsets[t] = ex;
        cursors[t] = ex;
    }
    if (t == 0) offsets[parts] = s[parts - 1];
}

template <int MODE>
__global__ void __launch_bounds__(PART_THREADS) part_scatter_kernel(const uint64_t* __restrict__ values, const uint32_t* __restrict__ validity,
                                                                    int64_t n, int is_f64, uint32_t parts, unsigned long long* cursors,
                                                                    uint64_t* __restrict__ out, uint64_t* const* __restrict__ outs,
                                                                    RangeSplit rs = RangeSplit{0, 1}, const uint8_t* __restrict__ pay_in = nullptr,
                                                                    uint8_t* const* __restrict__ pay_outs = nullptr, int pay_bytes = 0) {
    __shared__ uint64_t s_keys[PART_TILE];
    __shared__ uint64_t s_pay[MODE == PM_SPLIT ? PART_TILE : 1];
    __shared__ uint16_t s_part[PART_TILE];
    constexpr int NP = MODE == PM_SPLIT ? 64 : PART_MAX;  // the distributed sort has at most 64 destinations
    __shared__ uint32_t s_cnt[NP], s_off[NP];
    __shared__ unsigned long long s_gbase[NP];
    __shared__ uint32_t s_warp_tot[PART_THREADS / 32];
    const int64_t n_tiles = (n + PART_TILE - 1) / PART_TILE;
    const int per_thread = (int)(parts + PART_THREADS - 1) / PART_THREADS;  // buckets per thread in the scan (<= 4)
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        for (int i = threadIdx.x; i < (int)parts; i += PART_THREADS) s_cnt[i] = 0;
        __syncthreads();
        const int64_t base = tile * PART_TILE;
        uint64_t key[PART_KEYS_PER_THREAD];
        int part[PART_KEYS_PER_THREAD];
        uint32_t rank[PART_KEYS_PER_THREAD];
        load_classify<MODE>(values, validity, base, n, is_f64, parts, key, part, rs);
        // position inside the tile's run of its part. Few parts (the ranks of a shuffle): one returning shared atomic per
        // distinct part per warp instead of one per key
        const bool few = parts <= 64;
#pragma unroll
        for (int k = 0; k < PART_KEYS_PER_THREAD; ++k) {
            if (few) {
                const unsigned peers = __match_any_sync(0xffffffffu, part[k]);
                const int leader = __ffs(peers) - 1;
                uint32_t b0 = 0;
                if (part[k] >= 0 && (int)(threadIdx.x & 31) == leader) b0 = atomicAdd(&s_cnt[part[k]], (uint32_t)__popc(peers));
                b0 = __shfl_sync(0xffffffffu, b0, leader);
                rank[k] = b0 + (uint32_t)__popc(peers & ((1u << (threadIdx.x & 31)) - 1u));
            } else if (part[k] >= 0) {
                rank[k] = atomicAdd(&s_cnt[part[k]], 1u);
            }
        }
        __syncthreads();
        // exclusive scan of s_cnt over the buckets (thread t owns buckets t*per_thread ..), and one global
        // atomicAdd per non-empty bucket reserves this tile's run in the output
        {
            uint32_t loc[4], sum = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int b = threadIdx.x * per_thread + j;
                loc[j] = (j < per_thread && b < (int)parts) ? s_cnt[b] : 0;
                sum += loc[j];
            }
            uint32_t incl = sum;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
                if ((threadIdx.x & 31) >= d) incl += v;
            }
            if ((threadIdx.x & 31) == 31) s_warp_tot[threadIdx.x >> 5] = incl;
            __syncthreads();
            uint32_t warp_base = 0;
            for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) warp_base += s_warp_tot[w];
            uint32_t run = warp_base + incl - sum;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int b = threadIdx.x * per_thread + j;
                if (j < per_thread && b < (int)parts) {
                    s_off[b] = run;
                    if (loc[j]) s_gbase[b] = atomicAdd(&cursors[b], (unsigned long long)loc[j]);
                    run += loc[j];
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < PART_KEYS_PER_THREAD; ++k)
            if (part[k] >= 0) {
                const uint32_t pos = s_off[part[k]] + rank[k];
                s_keys[pos] = key[k];
                s_part[pos] = (uint16_t)part[k];
                if (MODE == PM_SPLIT && pay_bytes) {  // the payload of the same row travels with its key
                    const int64_t row = base + k * PART_THREADS + threadIdx.x;
                    s_pay[pos] = pay_bytes == 8 ? __ldg(reinterpret_cast<const unsigned long long*>(pay_in) + row)
                                                : (uint64_t)__ldg(reinterpret_cast<const uint32_t*>(pay_in) + row);
                }
            }
        __syncthreads();
        uint32_t total = 0;
        for (int w = 0; w < PART_THREADS / 32; ++w) total += s_warp_tot[w];
        // outs != nullptr: every part has its own destination buffer — the peer GPU's receive buffer, mapped through CUDA
        // IPC: the partition's output IS the all-to-all (the runs leave the SM as NVLink stores)
        for (uint32_t i = threadIdx.x; i < total; i += PART_THREADS) {
            const uint32_t b = s_part[i];
            uint64_t* dst = outs ? outs[b] : out;
            const unsigned long long gi = s_gbase[b] + (i - s_off[b]);
            dst[gi] = s_keys[i];
            if (MODE == PM_SPLIT && pay_bytes) {
                if (pay_bytes == 8) reinterpret_cast<uint64_t*>(pay_outs[b])[gi] = s_pay[i];
                else reinterpret_cast<uint32_t*>(pay_outs[b])[gi] = (uint32_t)s_pay[i];
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- per-bucket dedup ----
// Table reset between buckets. Plain stores (write-back, allocate in L2) instead of cudaMemsetAsync: the table is
// about to be hit by random atomics and should be L2-resident when the bucket's kernel starts.
__global__ void fill_kernel(uint4* __restrict__ p, size_t n16, uint32_t word) {
    const uint4 v = make_uint4(word, word, word, word);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}
static void fill_async(Engine& e, void* p, size_t bytes, uint32_t word, cudaStream_t stream = nullptr) {
    if (!stream) stream = e.stream;
    const size_t n16 = bytes / 16;
    const int grid = (int)std::min<size_t>((n16 + 255) / 256, (size_t)e.sm_count * 8);
    fill_kernel<<<std::max(grid, 1), 256, 0, stream>>>((uint4*)p, n16, word);
}
// bucket pipelines run side by side on this many streams, each with its own table: one bucket's kernel is a chain of
// dependent L2 atomics and does not fill the machine on its own
static int hash_lanes() {
    static const int v = [] {
        const char* e = getenv("TG_HASH_LANES");
        const int x = e ? atoi(e) : 0;
        return x >= 1 && x <= 4 ? x : 2;
    }();
    return v;
}

constexpr int BUCKET_ILP = 4;  // independent probe chains per thread (the loop is bound by L2 atomic latency)

// MASK: a key seen twice also goes into the repeated-key table R (key-level row verdicts)
template <bool MASK>
__global__ void __launch_bounds__(HASH_THREADS) insert_bucket_kernel(const uint64_t* __restrict__ keys, const unsigned long long* offsets,
                                                                     int bucket, unsigned long long* table, uint32_t mask, uint32_t* bits,
                                                                     HashCounters* ctr, RepTab R) {
    const int64_t begin = (int64_t)offsets[bucket], end = (int64_t)offsets[bucket + 1];
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned long long d = 0, dup = 0, ovf = 0;
    for (int64_t i0 = begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < end; i0 += stride * BUCKET_ILP) {
        uint64_t key[BUCKET_ILP];
        uint32_t slot[BUCKET_ILP];
        unsigned long long prev[BUCKET_ILP];
        bool live[BUCKET_ILP];
#pragma unroll
        for (int u = 0; u < BUCKET_ILP; ++u) {
            const int64_t i = i0 + u * stride;
            live[u] = i < end;
            key[u] = live[u] ? __ldg(keys + i) : 0ull;
        }
#pragma unroll
        for (int u = 0; u < BUCKET_ILP; ++u) {
            slot[u] = (uint32_t)fmix64(key[u]) & mask;
            if (live[u]) prev[u] = atomicCAS(&table[slot[u]], EMPTY64, (unsigned long long)key[u]);
        }
#pragma unroll
        for (int u = 0; u < BUCKET_ILP; ++u) {
            if (!live[u]) continue;
            for (uint32_t probes = 0;; ++probes) {
                if (prev[u] == EMPTY64) {
                    ++d;
                    break;
                }
                if (prev[u] == key[u]) {
                    const uint32_t bit = 1u << (slot[u] & 31);
                    if (!(atomicOr(&bits[slot[u] >> 5], bit) & bit)) {
                        ++dup;
                        if (MASK) rep_insert64(R, key[u]);
                    }
                    break;
                }
                if (probes >= mask) {
                    ovf = 1;
                    break;
                }
                slot[u] = (slot[u] + 1) & mask;
                prev[u] = atomicCAS(&table[slot[u]], EMPTY64, (unsigned long long)key[u]);
            }
        }
    }
    flush_counter_block(d, &ctr->distinct_nonnull);
    flush_counter_block(dup, &ctr->singles_minus);
    flush_counter_block(ovf, &ctr->overflow);
}

// FK: build the parent bucket's key set, then probe the child bucket
__global__ void __launch_bounds__(HASH_THREADS) build_bucket_kernel(const uint64_t* __restrict__ keys, const unsigned long long* offsets,
                                                                    int bucket, unsigned long long* table, uint32_t mask, HashCounters* ctr) {
    const int64_t begin = (int64_t)offsets[bucket], end = (int64_t)offsets[bucket + 1];
    unsigned long long ovf = 0;
    for (int64_t i = begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < end; i += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t key = keys[i];
        uint32_t slot = (uint32_t)fmix64(key) & mask;
        for (uint32_t probes = 0;; ++probes) {
            const unsigned long long prev = atomicCAS(&table[slot], EMPTY64, (unsigned long long)key);
            if (prev == EMPTY64 || prev == key) break;
            slot = (slot + 1) & mask;
            if (probes >= mask) {
                ovf = 1;
                break;
            }
        }
    }
    flush_counter(ovf, &ctr->overflow);
}

__global__ void __launch_bounds__(HASH_THREADS) probe_bucket_kernel(const uint64_t* __restrict__ keys, const unsigned long long* offsets,
                                                                    int bucket, const unsigned long long* __restrict__ table, uint32_t mask,
                                                                    int collect, unsigned long long* vkeys, uint64_t vmask,
                                                                    unsigned long long* examples, int max_examples, HashCounters* ctr) {
    const int64_t begin = (int64_t)offsets[bucket], end = (int64_t)offsets[bucket + 1];
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned long long viol = 0, dist = 0;
    for (int64_t i0 = begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < end; i0 += stride * BUCKET_ILP) {
        uint64_t key[BUCKET_ILP];
        uint32_t slot[BUCKET_ILP];
        unsigned long long v[BUCKET_ILP];
        bool live[BUCKET_ILP];
#pragma unroll
        for (int u = 0; u < BUCKET_ILP; ++u) {
            const int64_t i = i0 + u * stride;
            live[u] = i < end;
            key[u] = live[u] ? __ldg(keys + i) : 0ull;
        }
#pragma unroll
        for (int u = 0; u < BUCKET_ILP; ++u) {
            slot[u] = (uint32_t)fmix64(key[u]) & mask;
            v[u] = live[u] ? table[slot[u]] : 0ull;
        }
#pragma unroll
        for (int u = 0; u < BUCKET_ILP; ++u) {
            if (!live[u]) continue;
            bool found = false;
            while (true) {
                if (v[u] == key[u]) {
                    found = true;
                    break;
                }
                if (v[u] == EMPTY64) break;
                slot[u] = (slot[u] + 1) & mask;
                v[u] = table[slot[u]];
            }
            if (found) continue;
            ++viol;
            if (collect) {
                // dedupe the orphan keys; a full table (more distinct orphans than it was sized for) just stops
                // counting — the host sees violations > capacity / 2 and repeats the pass with an exact-size table
                uint64_t vs = (fmix64(key[u]) >> 20) & vmask;
                for (uint64_t probes = 0; probes <= vmask; ++probes) {
                    const unsigned long long prev = atomicCAS(&vkeys[vs], EMPTY64, (unsigned long long)key[u]);
                    if (prev == EMPTY64) {
                        ++dist;
                        const unsigned long long idx = atomicAdd(&ctr->n_examples, 1ull);
                        if (idx < (unsigned long long)max_examples) examples[idx] = key[u];
                        break;
                    }
                    if (prev == key[u]) break;
                    vs = (vs + 1) & vmask;
                }
            }
        }
    }
    flush_counter(viol, &ctr->violations);
    if (collect) flush_counter(dist, &ctr->distinct_all);
}

// ---------------------------------------------------------------- dense Int64 keys: bitmaps ----
// Keys such as auto-increment ids span a range not much larger than the row count. Then the "hash table" can be the
// identity: one bit per value of [min, max] for "seen" and one for "seen twice" — 2 x range/8 bytes, L2-resident up
// to 2^28 values, ONE returning atomicOr per key (126 G/s measured, tools/micro/atomics_bench.cu) and no
// partitioning pass at all. Exact, like the hash path; used when max - min < 2^28 and < 32 n.
struct MinMaxOut {
    long long mn, mx;
    unsigned long long n_valid;
    unsigned long long pad;
};
__global__ void __launch_bounds__(PART_THREADS) minmax_i64_kernel(const long long* __restrict__ values, const uint32_t* __restrict__ validity,
                                                                  int64_t n, MinMaxOut* out) {
    long long mn = INT64_MAX, mx = INT64_MIN;
    unsigned long long cnt = 0;
    const int64_t n_tiles = (n + PART_TILE - 1) / PART_TILE;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t base = tile * PART_TILE;
        long long v[PART_KEYS_PER_THREAD];
        uint32_t vw[PART_KEYS_PER_THREAD];
#pragma unroll
        for (int k = 0; k < PART_KEYS_PER_THREAD; ++k) {
            const int64_t row = base + k * PART_THREADS + threadIdx.x;
            const bool in = row < n;
            v[k] = in ? __ldg(values + row) : 0ll;
            vw[k] = in ? (validity ? __ldg(validity + (row >> 5)) : 0xffffffffu) : 0u;
        }
#pragma unroll
        for (int k = 0; k < PART_KEYS_PER_THREAD; ++k) {
            const int64_t row = base + k * PART_THREADS + threadIdx.x;
            if ((vw[k] >> (row & 31)) & 1u) {
                mn = min(mn, v[k]);
                mx = max(mx, v[k]);
                ++cnt;
            }
        }
    }
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, m));
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, m));
        cnt += __shfl_xor_sync(0xffffffffu, cnt, m);
    }
    if ((threadIdx.x & 31) == 0 && cnt) {
        atomicMin(&out->mn, mn);
        atomicMax(&out->mx, mx);
        atomicAdd(&out->n_valid, cnt);
    }
}

// number of set bits of a bitmap (distinct count after a non-returning build)
__global__ void bitmap_popcount_kernel(const uint4* __restrict__ bm, size_t n16, unsigned long long* out) {
    unsigned long long c = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) {
        const uint4 v = bm[i];
        c += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
    }
    flush_counter(c, out);
}

// min / max of a strided sample (every `stride`-th row): a range GUESS that lets the bitmap job run without a full
// min/max pass first; the job itself counts keys that fall outside and is repeated exactly when there are any
__global__ void __launch_bounds__(PART_THREADS) sample_minmax_i64_kernel(const long long* __restrict__ values, const uint32_t* __restrict__ validity,
                                                                         int64_t n, int64_t stride, MinMaxOut* out) {
    long long mn = INT64_MAX, mx = INT64_MIN;
    unsigned long long cnt = 0;
    const int64_t m = (n + stride - 1) / stride;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = i * stride;
        if (!row_valid(validity, row)) continue;
        const long long v = __ldg(values + row);
        mn = min(mn, v);
        mx = max(mx, v);
        ++cnt;
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, s));
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, s));
        cnt += __shfl_xor_sync(0xffffffffu, cnt, s);
    }
    if ((threadIdx.x & 31) == 0 && cnt) {
        atomicMin(&out->mn, mn);
        atomicMax(&out->mx, mx);
        atomicAdd(&out->n_valid, cnt);
    }
}

// mode 0: distinct / seen-twice counting; mode 1: build the parent set (non-returning OR); mode 2: probe
// MASK (mode 0): a key seen twice also goes into the repeated-key table R (key-level row verdicts)
template <int MODE, bool MASK = false>
__global__ void __launch_bounds__(PART_THREADS) dense_kernel(const long long* __restrict__ values, const uint32_t* __restrict__ validity,
                                                             int64_t n, long long lo, unsigned long long range, uint32_t* seen,
                                                             uint32_t* dup, unsigned long long* vkeys, uint64_t vmask,
                                                             unsigned long long* examples, int max_examples, HashCounters* ctr,
                                                             unsigned long long* nulls_out = nullptr, RepTab R = RepTab{}) {
    unsigned long long d = 0, dupk = 0, viol = 0, dist = 0, nulls = 0, special = 0, nulls_count = 0, oob = 0;
    const int64_t n_tiles = (n + PART_TILE - 1) / PART_TILE;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t base = tile * PART_TILE;
        long long v[PART_KEYS_PER_THREAD];
        uint32_t vw[PART_KEYS_PER_THREAD];
#pragma unroll
        for (int k = 0; k < PART_KEYS_PER_THREAD; ++k) {
            const int64_t row = base + k * PART_THREADS + threadIdx.x;
            const bool in = row < n;
            v[k] = in ? __ldg(values + row) : 0ll;
            vw[k] = in ? (validity ? __ldg(validity + (row >> 5)) : 0xffffffffu) : 0u;
        }
        uint32_t old[PART_KEYS_PER_THREAD];
        bool ok[PART_KEYS_PER_THREAD];
#pragma unroll
        for (int k = 0; k < PART_KEYS_PER_THREAD; ++k) {
            const int64_t row = base + k * PART_THREADS + threadIdx.x;
            ok[k] = (vw[k] >> (row & 31)) & 1u;
            nulls += (row < n) && !ok[k];
            nulls_count += (row < n) && !ok[k];
            const unsigned long long idx = ((unsigned long long)v[k] - (unsigned long long)lo);
            old[k] = 0;
            if (ok[k] && MODE != 2 && idx > range) {
                // outside the (guessed) key range: the bitmap cannot hold it; the host repeats the job with the exact range
                ++oob;
                ok[k] = false;
            }
            if (ok[k]) {
                const uint32_t bit = 1u << (idx & 31);
                if (MODE == 0) old[k] = atomicOr(&seen[idx >> 5], bit) & bit;
                else if (MODE == 1) atomicOr(&seen[idx >> 5], bit);  // result unused: RED.OR
                else old[k] = idx <= range ? (__ldg(&seen[idx >> 5]) & bit) : 0u;
            }
        }
#pragma unroll
        for (int k = 0; k < PART_KEYS_PER_THREAD; ++k) {
            if (!ok[k]) continue;
            if (MODE == 0) {
                if (!old[k]) {
                    ++d;
                } else {
                    const unsigned long long idx = ((unsigned long long)v[k] - (unsigned long long)lo);
                    const uint32_t bit = 1u << (idx & 31);
                    if (!(atomicOr(&dup[idx >> 5], bit) & bit)) {
                        ++dupk;
                        if (MASK) rep_insert64(R, (uint64_t)v[k]);
                    }
                }
            } else if (MODE == 2 && !old[k]) {
                ++viol;
                const uint64_t key = (uint64_t)v[k];
                if (key == EMPTY64) {  // the Int64 value -1 is the orphan table's EMPTY sentinel: counted apart
                    ++special;
                    continue;
                }
                uint64_t vs = (fmix64(key) >> 20) & vmask;
                for (uint64_t probes = 0; probes <= vmask; ++probes) {
                    const unsigned long long prev = atomicCAS(&vkeys[vs], EMPTY64, (unsigned long long)key);
                    if (prev == EMPTY64) {
                        ++dist;
                        const unsigned long long i = atomicAdd(&ctr->n_examples, 1ull);
                        if (i < (unsigned long long)max_examples) examples[i] = key;
                        break;
                    }
                    if (prev == key) break;
                    vs = (vs + 1) & vmask;
                }
            }
        }
    }
    if (MODE == 0) {
        flush_counter(d, &ctr->distinct_nonnull);
        flush_counter(dupk, &ctr->singles_minus);
    }
    if (MODE == 2) {
        flush_counter(viol, &ctr->violations);
        flush_counter(dist, &ctr->distinct_all);
        flush_counter(special, &ctr->special);
    }
    if (MODE != 1) flush_counter(nulls, &ctr->any_null_rows);
    if (MODE == 1 && nulls_out) flush_counter(nulls_count, nulls_out);
    if (MODE != 2) flush_counter(oob, &ctr->overflow);
}

// ================================================================== host side ==================
static size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static uint64_t pow2_at_least(uint64_t x, uint64_t lo) {
    uint64_t p = lo;
    while (p < x) p <<= 1;
    return p;
}
static int part_grid(Engine& e, int64_t n) {
    const int64_t tiles = (n + PART_TILE - 1) / PART_TILE;
    return (int)std::max<int64_t>(1, std::min<int64_t>(tiles, (int64_t)e.sm_count * 6));
}
static int bucket_grid(Engine& e, int64_t expected) {
    const int64_t blocks = (expected + HASH_THREADS - 1) / HASH_THREADS;
    return (int)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)e.sm_count * 8));
}
static uint32_t parts_for(int64_t n, int lanes = 1) {
    // `lanes` tables share the L2, so each bucket gets 1/lanes of the key budget
    const int64_t target = std::max<int64_t>(1024, bucket_target_keys() / lanes);
    return (uint32_t)std::min<uint64_t>(PART_MAX, pow2_at_least((uint64_t)((n + target - 1) / target), 1));
}

// device block: [hist parts][offsets parts+1][cursors parts][PartCounters], 256-byte aligned pieces
struct PartMeta {
    unsigned long long *hist, *offsets, *cursors;
    PartCounters* ctr;
    static size_t bytes() { return 3 * round_up((PART_MAX + 1) * 8, 256) + 256; }
    void bind(uint8_t* q) {
        hist = (unsigned long long*)q;
        offsets = (unsigned long long*)(q + round_up((PART_MAX + 1) * 8, 256));
        cursors = (unsigned long long*)(q + 2 * round_up((PART_MAX + 1) * 8, 256));
        ctr = (PartCounters*)(q + 3 * round_up((PART_MAX + 1) * 8, 256));
    }
};

// histogram + prefix + scatter of one column into `out` (capacity n keys); everything stays on the stream
template <int MODE>
static int partition_column(Engine& e, const Column& c, int64_t n, uint32_t parts, PartMeta& m, uint64_t* out) {
    TG_CUDA(cudaMemsetAsync(m.hist, 0, PartMeta::bytes(), e.stream));
    if (n == 0) {
        part_prefix_kernel<<<1, PART_MAX, 0, e.stream>>>(m.hist, parts, m.offsets, m.cursors);
        return 1;
    }
    const int grid = part_grid(e, n);
    const int is_f64 = c.dtype == TG_FLOAT64;
    part_hist_kernel<MODE><<<grid, PART_THREADS, 0, e.stream>>>((const uint64_t*)c.values.p, (const uint32_t*)c.validity.p, n, is_f64,
                                                               parts, m.hist, m.ctr);
    part_prefix_kernel<<<1, PART_MAX, 0, e.stream>>>(m.hist, parts, m.offsets, m.cursors);
    part_scatter_kernel<MODE><<<grid, PART_THREADS, 0, e.stream>>>((const uint64_t*)c.values.p, (const uint32_t*)c.validity.p, n, is_f64,
                                                                  parts, m.cursors, out, nullptr);
    TG_CUDA(cudaGetLastError());
    return 3;
}

struct MinMaxOut;
static bool minmax_i64(Engine& e, const Column& c, int64_t n, MinMaxOut& h, int& launches);

// The two halves of the partition as the push shuffle (comm.cpp) uses them: the histogram first — the ranks exchange the
// counts and derive where each part goes in its destination's receive buffer — then the scatter with those positions as
// cursors and one destination pointer per part (peer memory).
void push_partition_hist(Engine& e, const Column& c, int64_t n, int world, int64_t* counts, int64_t* n_nulls, int& launches,
                         const long long* range_min, unsigned long long range_span) {
    if (world < 1 || world > PART_MAX) throw Error(TG_ERR_INVALID_ARG, "world size must be in 1..1024");
    const size_t need = PartMeta::bytes() + 256;
    if (need > e.shuffle_cap) {
        TG_CUDA(cudaStreamSynchronize(e.stream));
        if (e.d_shuffle) TG_CUDA(cudaFree(e.d_shuffle));
        e.d_shuffle = nullptr;
        e.shuffle_cap = 0;
        TG_CUDA(cudaMalloc(&e.d_shuffle, need));
        e.shuffle_cap = need;
    }
    PartMeta m;
    m.bind(e.d_shuffle);
    TG_CUDA(cudaMemsetAsync(m.hist, 0, PartMeta::bytes(), e.stream));
    if (n > 0) {
        if (range_min)
            part_hist_kernel<PM_RANGE><<<part_grid(e, n), PART_THREADS, 0, e.stream>>>((const uint64_t*)c.values.p, (const uint32_t*)c.validity.p, n, 0,
                                                                                       (uint32_t)world, m.hist, m.ctr, RangeSplit::range(*range_min, range_span));
        else
            part_hist_kernel<PM_RANK><<<part_grid(e, n), PART_THREADS, 0, e.stream>>>((const uint64_t*)c.values.p, (const uint32_t*)c.validity.p, n,
                                                                                      c.dtype == TG_FLOAT64, (uint32_t)world, m.hist, m.ctr);
        TG_CUDA(cudaGetLastError());
        launches += 1;
    }
    std::vector<unsigned long long> h((size_t)world);
    PartCounters pc{};
    TG_CUDA(cudaMemcpyAsync(h.data(), m.hist, h.size() * 8, cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaMemcpyAsync(&pc, m.ctr, sizeof(pc), cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    for (int i = 0; i < world; ++i) counts[i] = (int64_t)h[i];
    *n_nulls = (int64_t)pc.nulls;
}
void push_partition_scatter(Engine& e, const Column& c, int64_t n, int world, const unsigned long long* first_index /* host, [world] */,
                            uint64_t* const* d_outs /* device array of world pointers */, int& launches, const long long* range_min,
                            unsigned long long range_span) {
    if (n <= 0) return;
    PartMeta m;
    m.bind(e.d_shuffle);
    TG_CUDA(cudaMemcpyAsync(m.cursors, first_index, (size_t)world * 8, cudaMemcpyHostToDevice, e.stream));
    if (range_min)
        part_scatter_kernel<PM_RANGE><<<part_grid(e, n), PART_THREADS, 0, e.stream>>>((const uint64_t*)c.values.p, (const uint32_t*)c.validity.p, n, 0,
                                                                                      (uint32_t)world, m.cursors, nullptr, d_outs,
                                                                                      RangeSplit::range(*range_min, range_span));
    else
        part_scatter_kernel<PM_RANK><<<part_grid(e, n), PART_THREADS, 0, e.stream>>>((const uint64_t*)c.values.p, (const uint32_t*)c.validity.p, n,
                                                                                     c.dtype == TG_FLOAT64, (uint32_t)world, m.cursors, nullptr, d_outs);
    TG_CUDA(cudaGetLastError());
    launches += 1;
}
// The distributed sort's exchange (ranks.cu / comm.cpp): raw 64-bit keys (no validity), destination = number of splitters
// below the key. d_splitters: world - 1 ascending keys on the device.
void split_partition_hist(Engine& e, const uint64_t* d_keys, int64_t n, int world, const uint64_t* d_splitters, int64_t* counts, int& launches) {
    const size_t need = PartMeta::bytes() + 256;
    if (need > e.shuffle_cap) {
        TG_CUDA(cudaStreamSynchronize(e.stream));
        if (e.d_shuffle) TG_CUDA(cudaFree(e.d_shuffle));
        e.d_shuffle = nullptr;
        e.shuffle_cap = 0;
        TG_CUDA(cudaMalloc(&e.d_shuffle, need));
        e.shuffle_cap = need;
    }
    PartMeta m;
    m.bind(e.d_shuffle);
    TG_CUDA(cudaMemsetAsync(m.hist, 0, PartMeta::bytes(), e.stream));
    if (n > 0) {
        part_hist_kernel<PM_SPLIT><<<part_grid(e, n), PART_THREADS, 0, e.stream>>>(d_keys, nullptr, n, 0, (uint32_t)world, m.hist, m.ctr,
                                                                                   RangeSplit{0, 1, d_splitters});
        TG_CUDA(cudaGetLastError());
        launches += 1;
    }
    std::vector<unsigned long long> h((size_t)world);
    TG_CUDA(cudaMemcpyAsync(h.data(), m.hist, h.size() * 8, cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    for (int i = 0; i < world; ++i) counts[i] = (int64_t)h[i];
}
void split_partition_scatter(Engine& e, const uint64_t* d_keys, const void* d_payload, int pay_bytes, int64_t n, int world,
                             const uint64_t* d_splitters, const unsigned long long* first_index, uint64_t* const* d_key_outs,
                             uint8_t* const* d_pay_outs, int& launches) {
    if (n <= 0) return;
    PartMeta m;
    m.bind(e.d_shuffle);
    TG_CUDA(cudaMemcpyAsync(m.cursors, first_index, (size_t)world * 8, cudaMemcpyHostToDevice, e.stream));
    part_scatter_kernel<PM_SPLIT><<<part_grid(e, n), PART_THREADS, 0, e.stream>>>(d_keys, nullptr, n, 0, (uint32_t)world, m.cursors, nullptr, d_key_outs,
                                                                                  RangeSplit{0, 1, d_splitters}, (const uint8_t*)d_payload, d_pay_outs,
                                                                                  pay_bytes);
    TG_CUDA(cudaGetLastError());
    launches += 1;
}

// min / max / valid count of an Int64 key column (the dense test of the range-partitioned shuffle)
// (large columns: from a strided 64 K-row sample — a partition only needs boundaries every rank agrees on; keys outside the
// sampled range go to the first / last rank, and the valid count is scaled up from the sample)
bool column_minmax_i64(Engine& e, const Column& c, int64_t n, long long* mn, long long* mx, unsigned long long* n_valid, int& launches) {
    MinMaxOut h{};
    if (n >= ((int64_t)1 << 22) && !getenv("TG_HASH_NO_GUESS")) {
        uint8_t* scr = e.scratch(256);
        MinMaxOut* d = (MinMaxOut*)scr;
        MinMaxOut init{INT64_MAX, INT64_MIN, 0, 0};
        TG_CUDA(cudaMemcpyAsync(d, &init, sizeof(init), cudaMemcpyHostToDevice, e.stream));
        const int64_t stride = std::max<int64_t>(1, n >> 16);
        sample_minmax_i64_kernel<<<64, PART_THREADS, 0, e.stream>>>((const long long*)c.values.p, (const uint32_t*)c.validity.p, n, stride, d);
        TG_CUDA(cudaGetLastError());
        ++launches;
        TG_CUDA(cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
        TG_CUDA(cudaStreamSynchronize(e.stream));
        *mn = h.mn;
        *mx = h.mx;
        *n_valid = h.n_valid * (unsigned long long)stride;
        return h.n_valid > 0;
    }
    const bool any = minmax_i64(e, c, n, h, launches);
    *mn = h.mn;
    *mx = h.mx;
    *n_valid = h.n_valid;
    return any;
}

bool distinct64_partitioned(Engine& e, const Column& c, int64_t n, Distinct64Result& r, int& launches, const RepTab* R) {
    const int lanes = hash_lanes();
    const uint32_t parts = parts_for(n, lanes);
    const uint64_t cap = pow2_at_least(((uint64_t)n + parts - 1) / parts * slots_factor(), 1024);
    const size_t keys_b = round_up((size_t)n * 8, 256), tab_b = cap * 8, bits_b = round_up(cap / 8, 256);
    uint8_t* scr = e.scratch(keys_b + (size_t)lanes * (tab_b + bits_b) + PartMeta::bytes() + 256);
    uint64_t* part_keys = (uint64_t*)scr;
    uint8_t* tables = scr + keys_b;
    PartMeta m;
    m.bind(tables + (size_t)lanes * (tab_b + bits_b));
    HashCounters* d_ctr = (HashCounters*)(tables + (size_t)lanes * (tab_b + bits_b) + PartMeta::bytes());
    TG_CUDA(cudaMemsetAsync(d_ctr, 0, sizeof(HashCounters), e.stream));
    if (R) rep_reset(e, *R);
    launches += partition_column<PM_BUCKET>(e, c, n, parts, m, part_keys);
    const int grid = bucket_grid(e, n / parts / BUCKET_ILP + 1);
    // fan out: lane l handles buckets l, l + lanes, .. on its own stream and table; fan back in before the read-back
    e.ensure_side_streams();
    TG_CUDA(cudaEventRecord(e.side_ev[4], e.stream));
    for (int l = 0; l < lanes; ++l) {
        cudaStream_t st = lanes == 1 ? e.stream : e.side[l];
        if (lanes > 1) TG_CUDA(cudaStreamWaitEvent(st, e.side_ev[4], 0));
        unsigned long long* table = (unsigned long long*)(tables + (size_t)l * (tab_b + bits_b));
        uint32_t* bits = (uint32_t*)(tables + (size_t)l * (tab_b + bits_b) + tab_b);
        for (uint32_t b = (uint32_t)l; b < parts; b += (uint32_t)lanes) {
            fill_async(e, table, tab_b, 0xFFFFFFFFu, st);
            fill_async(e, bits, bits_b, 0u, st);
            if (R) insert_bucket_kernel<true><<<grid, HASH_THREADS, 0, st>>>(part_keys, m.offsets, (int)b, table, (uint32_t)(cap - 1), bits, d_ctr, *R);
            else insert_bucket_kernel<false><<<grid, HASH_THREADS, 0, st>>>(part_keys, m.offsets, (int)b, table, (uint32_t)(cap - 1), bits, d_ctr, RepTab{});
            ++launches;
        }
        if (lanes > 1) {
            TG_CUDA(cudaEventRecord(e.side_ev[l], st));
            TG_CUDA(cudaStreamWaitEvent(e.stream, e.side_ev[l], 0));
        }
    }
    TG_CUDA(cudaGetLastError());
    HashCounters h{};
    PartCounters pc{};
    TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaMemcpyAsync(&pc, m.ctr, sizeof(pc), cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    if (h.overflow) return false;
    if (R && pc.special > 1) rep_mark(e, *R, EMPTY64);  // the Int64 value -1 never enters the bucket tables
    r.distinct = h.distinct_nonnull + (pc.special ? 1 : 0);
    r.dup_keys = h.singles_minus + (pc.special > 1 ? 1 : 0);
    r.nulls = pc.nulls;
    return true;
}

bool fk64_partitioned(Engine& e, const Column& child, int64_t nc, const Column& parent, int64_t np, int allow_nulls, int max_examples,
                      Fk64Result& r, int& launches, const VerdictOut* orphan_rows) {
    const uint32_t parts = parts_for(np);
    const uint64_t cap = pow2_at_least(((uint64_t)np + parts - 1) / parts * slots_factor(), 1024);
    const size_t ck_b = round_up((size_t)nc * 8, 256), pk_b = round_up((size_t)std::max<int64_t>(np, 1) * 8, 256), tab_b = cap * 8;
    // orphan keys are de-duplicated in the same pass into a small table (exact while violations <= FK_VCAP / 2)
    constexpr uint64_t FK_VCAP = 1u << 20;
    const size_t vk_b = FK_VCAP * 8, ex_b = round_up((size_t)std::max(max_examples, 1) * 8, 256);
    uint8_t* scr = e.scratch(ck_b + pk_b + tab_b + vk_b + ex_b + 2 * PartMeta::bytes() + 256);
    uint8_t* q = scr;
    uint64_t* ckeys = (uint64_t*)q; q += ck_b;
    uint64_t* pkeys = (uint64_t*)q; q += pk_b;
    unsigned long long* table = (unsigned long long*)q; q += tab_b;
    unsigned long long* vkeys0 = (unsigned long long*)q; q += vk_b;
    unsigned long long* d_ex0 = (unsigned long long*)q; q += ex_b;
    PartMeta mc, mp;
    mc.bind(q); q += PartMeta::bytes();
    mp.bind(q); q += PartMeta::bytes();
    HashCounters* d_ctr = (HashCounters*)q;
    TG_CUDA(cudaMemsetAsync(d_ctr, 0, sizeof(HashCounters), e.stream));
    TG_CUDA(cudaMemsetAsync(vkeys0, 0xFF, vk_b, e.stream));
    TG_CUDA(cudaMemsetAsync(d_ex0, 0, ex_b, e.stream));
    launches += partition_column<PM_BUCKET>(e, parent, np, parts, mp, pkeys);
    launches += partition_column<PM_BUCKET>(e, child, nc, parts, mc, ckeys);
    const int pgrid = bucket_grid(e, np / parts + 1), cgrid = bucket_grid(e, nc / parts / BUCKET_ILP + 1);
    auto pass = [&](unsigned long long* vkeys, uint64_t vmask, unsigned long long* examples) {
        for (uint32_t b = 0; b < parts; ++b) {
            fill_async(e, table, tab_b, 0xFFFFFFFFu);
            build_bucket_kernel<<<pgrid, HASH_THREADS, 0, e.stream>>>(pkeys, mp.offsets, (int)b, table, (uint32_t)(cap - 1), d_ctr);
            probe_bucket_kernel<<<cgrid, HASH_THREADS, 0, e.stream>>>(ckeys, mc.offsets, (int)b, table, (uint32_t)(cap - 1), 1, vkeys,
                                                                      vmask, examples, max_examples, d_ctr);
            launches += 2;
        }
        TG_CUDA(cudaGetLastError());
    };
    pass(vkeys0, FK_VCAP - 1, d_ex0);
    HashCounters h{};
    PartCounters hc{}, hp{};
    TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaMemcpyAsync(&hc, mc.ctr, sizeof(hc), cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaMemcpyAsync(&hp, mp.ctr, sizeof(hp), cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    if (h.overflow) return false;
    // the EMPTY-sentinel key (the Int64 value -1) never enters the tables: settle it here
    const bool special_orphan = hc.special > 0 && hp.special == 0;
    const uint64_t key_viol = h.violations + (special_orphan ? hc.special : 0);
    r.null_children = hc.nulls;
    r.violations = key_viol + (allow_nulls ? 0 : hc.nulls);
    r.distinct_violations = h.distinct_all;
    r.example_keys.clear();
    auto fetch_examples = [&](const unsigned long long* d_ex, uint64_t n_examples) {
        const size_t ne = (size_t)std::min<uint64_t>(n_examples, (uint64_t)std::max(max_examples, 0));
        r.example_keys.resize(ne);
        if (ne) TG_CUDA(cudaMemcpy(r.example_keys.data(), d_ex, ne * 8, cudaMemcpyDeviceToHost));
    };
    if (h.violations > FK_VCAP / 2) {
        // many orphans: repeat the pass with a de-duplication table sized from the now-known count
        const uint64_t vcap = pow2_at_least(h.violations * 2, 1024);
        uint8_t* extra = nullptr;
        TG_CUDA(cudaMalloc(&extra, vcap * 8));
        unsigned long long* vkeys = (unsigned long long*)extra;
        try {
            TG_CUDA(cudaMemsetAsync(vkeys, 0xFF, vcap * 8, e.stream));
            TG_CUDA(cudaMemsetAsync(d_ex0, 0, ex_b, e.stream));
            TG_CUDA(cudaMemsetAsync(d_ctr, 0, sizeof(HashCounters), e.stream));
            pass(vkeys, vcap - 1, d_ex0);
            TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
            TG_CUDA(cudaStreamSynchronize(e.stream));
            r.distinct_violations = h.distinct_all;
            fetch_examples(d_ex0, h.n_examples);
            if (orphan_rows) {
                fk_orphan_rows64(e, child, nc, vkeys, vcap - 1, 20, special_orphan, *orphan_rows, launches);
                TG_CUDA(cudaStreamSynchronize(e.stream));  // the pass reads `extra`, freed below
            }
        } catch (...) {
            cudaFree(extra);
            throw;
        }
        cudaFree(extra);
    } else {
        if (h.violations > 0) fetch_examples(d_ex0, h.n_examples);
        if (orphan_rows) fk_orphan_rows64(e, child, nc, h.violations > 0 ? vkeys0 : nullptr, FK_VCAP - 1, 20, special_orphan, *orphan_rows, launches);
    }
    if (special_orphan) {
        r.distinct_violations += 1;
        if ((int)r.example_keys.size() < max_examples) r.example_keys.push_back(EMPTY64);
    }
    return true;
}

void partition_keys_by_rank(Engine& e, const Column& c, int64_t n, int world, uint64_t** d_keys, int64_t* counts, int64_t* n_nulls,
                            int& launches) {
    if (world < 1 || world > PART_MAX) throw Error(TG_ERR_INVALID_ARG, "world size must be in 1..1024");
    const size_t keys_b = round_up((size_t)std::max<int64_t>(n, 1) * 8, 256);
    const size_t need = keys_b + PartMeta::bytes();
    if (need > e.shuffle_cap) {
        TG_CUDA(cudaStreamSynchronize(e.stream));
        if (e.d_shuffle) TG_CUDA(cudaFree(e.d_shuffle));
        e.d_shuffle = nullptr;
        e.shuffle_cap = 0;
        TG_CUDA(cudaMalloc(&e.d_shuffle, need));
        e.shuffle_cap = need;
    }
    PartMeta m;
    m.bind(e.d_shuffle + keys_b);
    launches += partition_column<PM_RANK>(e, c, n, (uint32_t)world, m, (uint64_t*)e.d_shuffle);
    std::vector<unsigned long long> off((size_t)world + 1);
    PartCounters pc{};
    TG_CUDA(cudaMemcpyAsync(off.data(), m.offsets, off.size() * 8, cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaMemcpyAsync(&pc, m.ctr, sizeof(pc), cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    for (int i = 0; i < world; ++i) counts[i] = (int64_t)(off[i + 1] - off[i]);
    *n_nulls = (int64_t)pc.nulls;
    *d_keys = (uint64_t*)e.d_shuffle;
}

// ---------------------------------------------------------------- dense-key front end ----
constexpr unsigned long long DENSE_MAX_RANGE = 1ull << 28;

// min / max / valid count of an Int64 column; returns false when it has no valid value
static bool minmax_i64(Engine& e, const Column& c, int64_t n, MinMaxOut& h, int& launches) {
    uint8_t* scr = e.scratch(256);
    MinMaxOut* d = (MinMaxOut*)scr;
    MinMaxOut init{INT64_MAX, INT64_MIN, 0, 0};
    TG_CUDA(cudaMemcpyAsync(d, &init, sizeof(init), cudaMemcpyHostToDevice, e.stream));
    if (n > 0) {
        minmax_i64_kernel<<<part_grid(e, n), PART_THREADS, 0, e.stream>>>((const long long*)c.values.p, (const uint32_t*)c.validity.p, n, d);
        TG_CUDA(cudaGetLastError());
        ++launches;
    }
    TG_CUDA(cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    return h.n_valid > 0;
}
static bool dense_enough(const MinMaxOut& h) {
    const unsigned long long range = (unsigned long long)h.mx - (unsigned long long)h.mn;
    return range < DENSE_MAX_RANGE && range <= 32ull * h.n_valid + 4096ull;
}

// one bitmap pass over [lo, lo + range]; returns the counters (overflow = keys outside the range)
static HashCounters dense_distinct_pass(Engine& e, const Column& c, int64_t n, bool need_singles, long long lo, unsigned long long range,
                                        int& launches, const RepTab* R) {
    const size_t bm_b = round_up((size_t)(range / 32 + 1) * 4, 256);
    uint8_t* scr = e.scratch(2 * bm_b + 256);
    uint32_t* seen = (uint32_t*)scr;
    uint32_t* dup = (uint32_t*)(scr + bm_b);
    HashCounters* d_ctr = (HashCounters*)(scr + 2 * bm_b);
    if (need_singles) {
        // one RETURNING atomicOr per key: the old bit tells first from repeated occurrence
        fill_async(e, scr, 2 * bm_b + 256, 0u);
        if (R) {
            rep_reset(e, *R);
            dense_kernel<0, true><<<part_grid(e, n), PART_THREADS, 0, e.stream>>>((const long long*)c.values.p, (const uint32_t*)c.validity.p, n, lo,
                                                                                  range, seen, dup, nullptr, 0, nullptr, 0, d_ctr, nullptr, *R);
        } else {
            dense_kernel<0><<<part_grid(e, n), PART_THREADS, 0, e.stream>>>((const long long*)c.values.p, (const uint32_t*)c.validity.p, n, lo, range,
                                                                           seen, dup, nullptr, 0, nullptr, 0, d_ctr);
        }
        launches += 2;
    } else {
        // only COUNT(DISTINCT) is wanted: non-returning ORs (190 vs 126 G/s in L2), then count the set bits
        fill_async(e, seen, bm_b, 0u);
        fill_async(e, d_ctr, 256, 0u);
        dense_kernel<1><<<part_grid(e, n), PART_THREADS, 0, e.stream>>>((const long long*)c.values.p, (const uint32_t*)c.validity.p, n, lo, range,
                                                                       seen, nullptr, nullptr, 0, nullptr, 0, d_ctr, &d_ctr->any_null_rows);
        const size_t n16 = bm_b / 16;
        bitmap_popcount_kernel<<<(int)std::max<size_t>(1, std::min<size_t>((n16 + 255) / 256, (size_t)e.sm_count * 8)), 256, 0, e.stream>>>(
            (const uint4*)seen, n16, &d_ctr->distinct_nonnull);
        launches += 4;
    }
    TG_CUDA(cudaGetLastError());
    HashCounters h{};
    TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    return h;
}

bool distinct64_dense(Engine& e, const Column& c, int64_t n, bool need_singles, Distinct64Result& r, int& launches, const RepTab* R) {
    if (c.dtype != TG_INT64 || getenv("TG_HASH_NO_DENSE")) return false;
    need_singles = need_singles || R;  // the row verdicts need the 1 -> 2 transitions of the seen-twice map
    auto fill_result = [&](const HashCounters& h) {
        r.distinct = h.distinct_nonnull;
        r.dup_keys = need_singles ? h.singles_minus : 0;  // unused by the slots of this plan when !need_singles
        r.nulls = h.any_null_rows;
    };
    // 1. optimistic: guess the key range from a strided 64 K sample, padded by 1/16 of its width on both sides. For
    //    ids / surrogate keys the guess holds and the min/max pass over the whole column is saved.
    static const int64_t guess_min_rows = [] {
        const char* ev = getenv("TG_HASH_GUESS_MIN_ROWS");
        const long long x = ev ? atoll(ev) : 0;
        return x > 0 ? (int64_t)x : (int64_t)1 << 22;
    }();
    if (n >= guess_min_rows && !getenv("TG_HASH_NO_GUESS")) {
        uint8_t* scr = e.scratch(256);
        MinMaxOut* d = (MinMaxOut*)scr;
        MinMaxOut init{INT64_MAX, INT64_MIN, 0, 0}, g{};
        TG_CUDA(cudaMemcpyAsync(d, &init, sizeof(init), cudaMemcpyHostToDevice, e.stream));
        const int64_t stride = std::max<int64_t>(1, n >> 16);
        sample_minmax_i64_kernel<<<64, PART_THREADS, 0, e.stream>>>((const long long*)c.values.p, (const uint32_t*)c.validity.p, n, stride, d);
        TG_CUDA(cudaGetLastError());
        ++launches;
        TG_CUDA(cudaMemcpyAsync(&g, d, sizeof(g), cudaMemcpyDeviceToHost, e.stream));
        TG_CUDA(cudaStreamSynchronize(e.stream));
        if (g.n_valid > 0) {
            const unsigned long long w = (unsigned long long)g.mx - (unsigned long long)g.mn;
            // the column's range is at least the sample's and it holds at most n valid keys: a sample that is not dense
            // settles it without the min/max pass over the whole column
            if (w >= DENSE_MAX_RANGE || w > 32ull * (unsigned long long)n + 4096ull) return false;
            const unsigned long long pad = w / 16 + 4096;
            // keep lo / hi inside i64 (the wrap-around arithmetic of the kernel handles the rest)
            const long long lo = g.mn < INT64_MIN + (long long)pad ? INT64_MIN : g.mn - (long long)pad;
            const long long hi = g.mx > INT64_MAX - (long long)pad ? INT64_MAX : g.mx + (long long)pad;
            const unsigned long long range = (unsigned long long)hi - (unsigned long long)lo;
            if (range < DENSE_MAX_RANGE && range <= 32ull * (unsigned long long)n + 4096ull) {
                const HashCounters h = dense_distinct_pass(e, c, n, need_singles, lo, range, launches, R);
                if (h.overflow == 0) {
                    fill_result(h);
                    return true;
                }
            }
        }
    }
    // 2. exact range from a full min/max pass
    MinMaxOut mm{};
    if (!minmax_i64(e, c, n, mm, launches)) {
        r = Distinct64Result{0, 0, (uint64_t)n};
        return true;
    }
    if (!dense_enough(mm)) return false;
    const unsigned long long range = (unsigned long long)mm.mx - (unsigned long long)mm.mn;
    fill_result(dense_distinct_pass(e, c, n, need_singles, mm.mn, range, launches, R));
    return true;
}

bool fk64_dense(Engine& e, const Column& child, int64_t nc, const Column& parent, int64_t np, int allow_nulls, int max_examples,
                Fk64Result& r, int& launches, const VerdictOut* orphan_rows) {
    if (child.dtype != TG_INT64 || parent.dtype != TG_INT64 || getenv("TG_HASH_NO_DENSE")) return false;
    MinMaxOut mm{};
    const bool have_parent = minmax_i64(e, parent, np, mm, launches);
    if (have_parent && !dense_enough(mm)) return false;
    const unsigned long long range = have_parent ? (unsigned long long)mm.mx - (unsigned long long)mm.mn : 0ull;
    const size_t bm_b = round_up((size_t)(range / 32 + 1) * 4, 256);
    constexpr uint64_t FK_VCAP = 1u << 20;
    const size_t vk_b = FK_VCAP * 8, ex_b = round_up((size_t)std::max(max_examples, 1) * 8, 256);
    uint8_t* scr = e.scratch(bm_b + vk_b + ex_b + 256);
    uint32_t* seen = (uint32_t*)scr;
    unsigned long long* vkeys0 = (unsigned long long*)(scr + bm_b);
    unsigned long long* d_ex = (unsigned long long*)(scr + bm_b + vk_b);
    HashCounters* d_ctr = (HashCounters*)(scr + bm_b + vk_b + ex_b);
    fill_async(e, seen, bm_b, 0u);
    fill_async(e, vkeys0, vk_b, 0xFFFFFFFFu);
    fill_async(e, d_ex, ex_b + 256, 0u);
    launches += 3;
    if (have_parent) {
        dense_kernel<1><<<part_grid(e, np), PART_THREADS, 0, e.stream>>>((const long long*)parent.values.p, (const uint32_t*)parent.validity.p, np,
                                                                        mm.mn, range, seen, nullptr, nullptr, 0, nullptr, 0, d_ctr);
        ++launches;
    }
    // an empty parent set: lo = 0, range = 0 and an all-zero bitmap -> every child key is an orphan
    auto probe = [&](unsigned long long* vkeys, uint64_t vmask) {
        dense_kernel<2><<<part_grid(e, nc), PART_THREADS, 0, e.stream>>>((const long long*)child.values.p, (const uint32_t*)child.validity.p, nc,
                                                                        have_parent ? mm.mn : 0, range, seen, nullptr, vkeys, vmask, d_ex,
                                                                        max_examples, d_ctr);
        TG_CUDA(cudaGetLastError());
        ++launches;
    };
    probe(vkeys0, FK_VCAP - 1);
    HashCounters h{};
    TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    if (h.violations > FK_VCAP / 2) {
        const uint64_t vcap = pow2_at_least(h.violations * 2, 1024);
        uint8_t* extra = nullptr;
        TG_CUDA(cudaMalloc(&extra, vcap * 8));
        try {
            fill_async(e, extra, vcap * 8, 0xFFFFFFFFu);
            fill_async(e, d_ex, ex_b + 256, 0u);
            probe((unsigned long long*)extra, vcap - 1);
            TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
            TG_CUDA(cudaStreamSynchronize(e.stream));
            if (orphan_rows) {
                fk_orphan_rows64(e, child, nc, (const unsigned long long*)extra, vcap - 1, 20, h.special > 0, *orphan_rows, launches);
                TG_CUDA(cudaStreamSynchronize(e.stream));  // the pass reads `extra`, freed below
            }
        } catch (...) {
            cudaFree(extra);
            throw;
        }
        cudaFree(extra);
    } else if (orphan_rows) {
        fk_orphan_rows64(e, child, nc, h.violations > h.special ? vkeys0 : nullptr, FK_VCAP - 1, 20, h.special > 0, *orphan_rows, launches);
    }
    r.null_children = h.any_null_rows;
    r.violations = h.violations + (allow_nulls ? 0 : h.any_null_rows);
    r.distinct_violations = h.distinct_all + (h.special ? 1 : 0);
    const size_t ne = (size_t)std::min<uint64_t>(h.n_examples, (uint64_t)std::max(max_examples, 0));
    r.example_keys.resize(ne);
    if (ne) TG_CUDA(cudaMemcpy(r.example_keys.data(), d_ex, ne * 8, cudaMemcpyDeviceToHost));
    if (h.special && (int)r.example_keys.size() < max_examples) r.example_keys.push_back(EMPTY64);
    return true;
}

}  // namespace tg
