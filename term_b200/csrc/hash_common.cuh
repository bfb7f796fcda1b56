// Shared device helpers of the hash jobs (hashing.cu: single-table path for small inputs, Utf8 / composite keys and
// grouped counts; hashpart.cu: radix-partitioned path for large Int64 / Float64 key columns and the multi-GPU shuffle).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace tg {

constexpr unsigned long long EMPTY64 = 0xFFFFFFFFFFFFFFFFull;
constexpr int HASH_THREADS = 256;

__host__ __device__ __forceinline__ uint64_t fmix64(uint64_t k) {
    k ^= k >> 33;
    k *= 0xff51afd7ed558ccdull;
    k ^= k >> 33;
    k *= 0xc4ceb9fe1a85ec53ull;
    k ^= k >> 33;
    return k;
}
__host__ __device__ __forceinline__ uint64_t canon_f64(uint64_t bits) {
    // -0.0 == +0.0 and all NaNs compare as one value when grouping
    if ((bits << 1) == 0) return 0;
    if ((bits & 0x7ff0000000000000ull) == 0x7ff0000000000000ull && (bits & 0x000fffffffffffffull)) return 0x7ff8000000000000ull;
    return bits;
}
__device__ __forceinline__ bool row_valid(const uint32_t* validity, int64_t row) {
    return !validity || ((validity[row >> 5] >> (row & 31)) & 1u);
}

// How the 64 hash bits of a key are spent (disjoint fields, so the levels are independent):
//   bits  0..31  slot inside a (bucket-local) hash table
//   bits 32..41  local radix bucket (<= 1024 buckets per GPU)
//   bits 42..63  destination rank of the multi-GPU shuffle: (top22 * world) >> 22
__host__ __device__ __forceinline__ uint32_t hash_bucket(uint64_t h, uint32_t pmask) { return (uint32_t)(h >> 32) & pmask; }
__host__ __device__ __forceinline__ uint32_t hash_rank(uint64_t h, uint32_t world) { return (uint32_t)(((h >> 42) * world) >> 22); }

struct HashCounters {
    unsigned long long distinct_all;      // groups, NULL as a value
    unsigned long long distinct_nonnull;  // groups whose key has no NULL component
    unsigned long long singles_plus;      // +1 on first insert
    unsigned long long singles_minus;     // +1 on second insert
    unsigned long long any_null_rows;
    unsigned long long special;           // rows whose exact key equals the EMPTY sentinel (path A)
    unsigned long long violations;        // FK
    unsigned long long null_children;     // FK
    unsigned long long n_examples;
    unsigned long long overflow;          // a bucket table filled up (skewed hash): the caller falls back
    unsigned long long pad[6];
};

// block-level reduction of per-thread counters, one atomic per counter per warp
__device__ __forceinline__ void flush_counter(unsigned long long v, unsigned long long* dst) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(dst, v);
}

// the same with ONE global atomic per block (every thread of the block must call it): the bucket kernels are launched per
// bucket with ~1000 blocks each, and a warp-granular flush made thousands of same-address atomics the tail of every launch
__device__ __forceinline__ void flush_counter_block(unsigned long long v, unsigned long long* dst) {
    __shared__ unsigned long long s_part[32];
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
    const int warp = threadIdx.x >> 5, n_warps = (blockDim.x + 31) >> 5;
    __syncthreads();  // (s_part may still be read by the previous counter's flush)
    if ((threadIdx.x & 31) == 0) s_part[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < n_warps; ++w) t += s_part[w];
        if (t) atomicAdd(dst, t);
    }
}

// ---- 128-bit fingerprints of Utf8 / composite keys ----
struct Fp {
    uint64_t h1, h2;
};
constexpr uint64_t NULL_TAG1 = 0x9ae16a3b2f90404full, NULL_TAG2 = 0xc3a5c85c97cb3127ull;

__device__ __forceinline__ void fp_combine(Fp& acc, uint64_t a, uint64_t b, bool first) {
    if (first) {
        acc.h1 = fmix64(a ^ 0x2545f4914f6cdd1dull);
        acc.h2 = fmix64(b + 0x9e3779b97f4a7c15ull);
    } else {
        acc.h1 = fmix64(acc.h1 * 0x9e3779b97f4a7c15ull + a);
        acc.h2 = fmix64((acc.h2 ^ b) * 0xd6e8feb86659fd93ull + 0x632be59bd9b4e019ull);
    }
}


struct Table128 {
    unsigned long long* h1;
    unsigned long long* h2;
    uint32_t* counts;
    uint64_t mask;
};

// find-or-insert a fingerprint; returns the slot and whether this call created it
__device__ __forceinline__ uint64_t upsert128(const Table128& t, Fp f, bool& created) {
    uint64_t a = f.h1 == EMPTY64 ? 0 : f.h1, b = f.h2 == EMPTY64 ? 0 : f.h2;
    uint64_t slot = (a ^ (b >> 32)) & t.mask;
    created = false;
    while (true) {
        const unsigned long long prev = atomicCAS(&t.h1[slot], EMPTY64, (unsigned long long)a);
        if (prev == EMPTY64) {
            // claimed: publish the second word
            atomicExch(&t.h2[slot], (unsigned long long)b);
            created = true;
            return slot;
        }
        if (prev == a) {
            unsigned long long v;
            do {
                v = *reinterpret_cast<volatile unsigned long long*>(&t.h2[slot]);
            } while (v == EMPTY64);
            if (v == b) return slot;
        }
        slot = (slot + 1) & t.mask;
    }
}

// ---- key-level row verdicts (tg_plan_request_key_rows) ----
// fmix64 is a bijection; its inverse turns the hashes the sorted-bucket path de-duplicates back into keys
__host__ __device__ __forceinline__ uint64_t fmix64_inv(uint64_t h) {
    h ^= h >> 33;
    h *= 0x9cb4b2f8129337dbull;  // inverse of 0xc4ceb9fe1a85ec53 mod 2^64
    h ^= h >> 33;
    h *= 0x4f74430c22a54005ull;  // inverse of 0xff51afd7ed558ccd mod 2^64
    h ^= h >> 33;
    return h;
}

// Repeated-key table R: every key that occurs in at least two rows, inserted by the counting kernels at the moment a key's
// count goes from 1 to 2 (so each key once), then the lowest row holding it (atomicMin by the row pass). 64-bit keys are
// the canonical values; Utf8 / composite keys the two fingerprint words (h2 != nullptr). The 64-bit key equal to the EMPTY
// word (the Int64 value -1) has its own cell: empty_key[0] = 1 when it is repeated, empty_key[1] = its lowest row.
// R never holds more than half its slots: an insert first claims one of those places (`fill`), and past them the counting
// pass inserts nothing more. The host, which knows the repeated-key count, then repeats the job once with R sized from it.
// So no insert probes a full or crowded table, whatever the number of repeated keys.
struct RepTab {
    unsigned long long* h1 = nullptr;  // nullptr: no key is repeated (every row is the first of its key)
    unsigned long long* h2 = nullptr;
    unsigned long long* minrow = nullptr;
    unsigned long long* empty_key = nullptr;
    unsigned long long* fill = nullptr;  // places claimed so far
    uint64_t mask = 0;
};
__device__ __forceinline__ uint64_t rep_home(uint64_t a, uint64_t b) { return fmix64(a ^ 0x9e3779b97f4a7c15ull ^ (b << 1)); }
// (the plain load first: once R is at half, the remaining repeated keys of the pass read one L2-resident word, no atomic)
__device__ __forceinline__ bool rep_claim(const RepTab& R) {
    const unsigned long long half = (R.mask + 1) / 2;
    return *reinterpret_cast<volatile unsigned long long*>(R.fill) < half && atomicAdd(R.fill, 1ull) < half;
}

__device__ __forceinline__ void rep_insert64(const RepTab& R, uint64_t key) {
    if (key == EMPTY64) {
        R.empty_key[0] = 1ull;
        return;
    }
    if (!rep_claim(R)) return;
    uint64_t slot = rep_home(key, 0) & R.mask;
    for (uint64_t probes = 0; probes <= R.mask; ++probes) {
        if (atomicCAS(&R.h1[slot], EMPTY64, (unsigned long long)key) == EMPTY64) return;
        slot = (slot + 1) & R.mask;
    }
}
__device__ __forceinline__ void rep_insert128(const RepTab& R, Fp f) {
    const uint64_t a = f.h1 == EMPTY64 ? 0 : f.h1, b = f.h2;  // (a free slot is h1 == EMPTY, as in upsert128)
    if (!rep_claim(R)) return;
    uint64_t slot = rep_home(a, b) & R.mask;
    for (uint64_t probes = 0; probes <= R.mask; ++probes) {
        if (atomicCAS(&R.h1[slot], EMPTY64, (unsigned long long)a) == EMPTY64) {
            R.h2[slot] = b;  // read only by the row passes, which are later launches
            return;
        }
        slot = (slot + 1) & R.mask;
    }
}
// the min-row cell of a key, nullptr when it is not repeated
__device__ __forceinline__ unsigned long long* rep_cell64(const RepTab& R, uint64_t key) {
    if (!R.h1) return nullptr;
    if (key == EMPTY64) return R.empty_key[0] ? &R.empty_key[1] : nullptr;
    uint64_t slot = rep_home(key, 0) & R.mask;
    for (uint64_t probes = 0; probes <= R.mask; ++probes) {
        const unsigned long long v = R.h1[slot];
        if (v == key) return &R.minrow[slot];
        if (v == EMPTY64) return nullptr;
        slot = (slot + 1) & R.mask;
    }
    return nullptr;
}
__device__ __forceinline__ unsigned long long* rep_cell128(const RepTab& R, Fp f) {
    if (!R.h1) return nullptr;
    const uint64_t a = f.h1 == EMPTY64 ? 0 : f.h1, b = f.h2;
    uint64_t slot = rep_home(a, b) & R.mask;
    for (uint64_t probes = 0; probes <= R.mask; ++probes) {
        const unsigned long long v = R.h1[slot];
        if (v == EMPTY64) return nullptr;
        if (v == a && R.h2[slot] == b) return &R.minrow[slot];
        slot = (slot + 1) & R.mask;
    }
    return nullptr;
}

// Output words of one key-level verdict array (Arrow Boolean: values, and validity or nullptr)
struct VerdictOut {
    uint32_t* values = nullptr;
    uint32_t* validity = nullptr;
};
// One warp stores the 32-row word w: lane l holds row 32 w + l (bits past the last row are false)
__device__ __forceinline__ void store_verdict_word(int64_t w, bool bit, bool valid, const VerdictOut& o) {
    const uint32_t vb = __ballot_sync(0xffffffffu, bit && valid), vv = __ballot_sync(0xffffffffu, valid);
    if ((threadIdx.x & 31) == 0) {
        if (o.values) o.values[w] = vb;
        if (o.validity) o.validity[w] = vv;
    }
}

}  // namespace tg
