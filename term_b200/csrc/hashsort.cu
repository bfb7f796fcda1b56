// K3 (large sparse key columns) — sorted-bucket de-duplication of a single Int64 / Float64 key column.
//
// Replaces  COUNT(DISTINCT c) / GROUP BY c HAVING COUNT(*) = 1                   constraints/uniqueness.rs:549-718
// for key columns that are neither dense (bitmap path, hashpart.cu) nor small (single table, hashing.cu).
//
// The L2-resident bucket tables of hashpart.cu pay one global atomicCAS per key (~110 G/s at best, and one small launch
// per bucket). Here no key ever meets a global atomic:
//   1. hs_prep_kernel    valid rows -> h = fmix64(canonical key), compacted (order is irrelevant). fmix64 is a BIJECTION
//                        on 64 bits, so distinct keys <=> distinct h and the counts are exact; NULLs are counted, the one
//                        key whose hash equals the table's EMPTY word is counted aside.
//   2. two (three above 2^27 rows) passes of the onesweep radix sort (radix_sort.cu) over the LOW 16 (24) bits of h:
//                        65536 (16 M) hash buckets of <= ~2000 keys, contiguous in memory. Equal keys share a bucket.
//   3. hs_dedup_kernel   CTAs walk the bucket-sorted array in fixed chunks; a CTA owns the buckets whose FIRST key lies
//                        in its chunk (it reads on past the chunk's end until the last of them closes; the keys of a
//                        bucket that began earlier are left to its owner) and de-duplicates them in a shared-memory
//                        table (64-bit CAS in shared memory, a 1-bit "seen twice" map) — every key is read once, from
//                        a coalesced stream.
// A bucket far beyond its expected size (a hot key: > HS_MAX_TAIL_ROUNDS * HS_THREADS copies) or a table that fills up
// raises a flag and the caller falls back to the partitioned path, which handles both.
#include <algorithm>
#include <cstdlib>

#include "hash_common.cuh"
#include "hashpart.hpp"
#include "radix_sort.cuh"

namespace tg {

#ifndef TG_HS_THREADS
#define TG_HS_THREADS 512
#define TG_HS_CHUNK 2048
#define TG_HS_SLOTS 8192
#define TG_HS_SPEC 5
#endif
constexpr int HS_THREADS = TG_HS_THREADS, HS_WARPS = HS_THREADS / 32;
constexpr int HS_KEYS = 4096 / HS_THREADS;       // rows per thread per tile of the prep kernel (128 (row group, warp) counts per tile)
constexpr int HS_TILE = HS_THREADS * HS_KEYS;
constexpr int HS_CHUNK = TG_HS_CHUNK;            // nominal keys per chunk of the dedup kernel
constexpr int HS_SLOTS = TG_HS_SLOTS;            // shared table: chunk + the tail of its last bucket at load <= ~0.5
constexpr int HS_SPEC = TG_HS_SPEC;              // rounds of HS_THREADS keys past the chunk that are loaded speculatively
constexpr int HS_MAX_TAIL_ROUNDS = (128 << 10) / HS_THREADS;  // a bucket that runs > 128 K keys past its chunk is not a hash bucket: skew

struct HsCounters {
    unsigned long long n_valid;   // keys written by the prep kernel
    unsigned long long nulls;
    unsigned long long special;   // valid rows whose hash is the EMPTY word
    unsigned long long distinct;
    unsigned long long dup_keys;  // keys seen at least twice
    unsigned long long overflow;
    unsigned long long skew;
    unsigned long long pad;
};

static size_t hs_round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

__global__ void __launch_bounds__(HS_THREADS) hs_prep_kernel(const uint64_t* __restrict__ values, const uint32_t* __restrict__ validity, int64_t n,
                                                             int is_f64, uint64_t* __restrict__ out, HsCounters* ctr,
                                                             unsigned long long* __restrict__ hist, int n_passes) {
    __shared__ uint32_t s_cnt[HS_KEYS * HS_WARPS];  // [k][warp]: kept rows of the warp's k-th row group, then their offsets
    __shared__ unsigned long long s_base;
    __shared__ uint32_t s_hist[3][RS_BINS];         // digit counts of the sort that follows (a block sees < 2^32 keys)
    for (int i = threadIdx.x; i < 3 * RS_BINS; i += HS_THREADS) (&s_hist[0][0])[i] = 0;
    __syncthreads();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned lt = (1u << lane) - 1u;
    unsigned long long nulls = 0, special = 0;
    const int64_t n_tiles = (n + HS_TILE - 1) / HS_TILE;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t base = tile * HS_TILE;
        uint64_t h[HS_KEYS];
        uint32_t vw[HS_KEYS];
#pragma unroll
        for (int k = 0; k < HS_KEYS; ++k) {
            const int64_t row = base + k * HS_THREADS + tid;
            const bool in = row < n;
            h[k] = in ? __ldg(values + row) : 0ull;
            vw[k] = in ? (validity ? __ldg(validity + (row >> 5)) : 0xffffffffu) : 0u;
        }
        uint32_t keep = 0, pos[HS_KEYS];
#pragma unroll
        for (int k = 0; k < HS_KEYS; ++k) {
            const int64_t row = base + k * HS_THREADS + tid;
            bool valid = (vw[k] >> (row & 31)) & 1u;
            if (row < n && !valid) ++nulls;
            h[k] = fmix64(is_f64 ? canon_f64(h[k]) : h[k]);
            if (valid && h[k] == EMPTY64) {
                ++special;
                valid = false;
            }
            if (valid) {
                atomicAdd(&s_hist[0][h[k] & 255u], 1u);
                atomicAdd(&s_hist[1][(h[k] >> 8) & 255u], 1u);
                if (n_passes > 2) atomicAdd(&s_hist[2][(h[k] >> 16) & 255u], 1u);
            }
            const unsigned m = __ballot_sync(0xffffffffu, valid);
            if (lane == 0) s_cnt[k * HS_WARPS + warp] = (uint32_t)__popc(m);
            pos[k] = (uint32_t)__popc(m & lt);
            keep |= (valid ? 1u : 0u) << k;
        }
        __syncthreads();
        if (warp == 0) {  // exclusive scan of the HS_KEYS * HS_WARPS = 128 counts, four per lane
            uint32_t c[4], sum = 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                c[i] = s_cnt[lane * 4 + i];
                sum += c[i];
            }
            uint32_t x = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= o) x += y;
            }
            uint32_t run = x - sum;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                s_cnt[lane * 4 + i] = run;
                run += c[i];
            }
            if (lane == 31) s_base = atomicAdd(&ctr->n_valid, (unsigned long long)x);
        }
        __syncthreads();
        const unsigned long long b = s_base;
#pragma unroll
        for (int k = 0; k < HS_KEYS; ++k)
            if ((keep >> k) & 1u) out[b + s_cnt[k * HS_WARPS + warp] + pos[k]] = h[k];
        __syncthreads();
    }
    for (int i = tid; i < n_passes * RS_BINS; i += HS_THREADS) {
        const uint32_t v = (&s_hist[0][0])[i];
        if (v) atomicAdd(&hist[i], (unsigned long long)v);
    }
    flush_counter_block(nulls, &ctr->nulls);
    flush_counter_block(special, &ctr->special);
}

struct HsLocal {
    uint32_t distinct, dups, overflow;
};
// MASK: a key seen twice also goes into the repeated-key table R, as the key its hash came from
template <bool MASK>
__device__ __forceinline__ void hs_insert(unsigned long long* tab, uint32_t* twice, uint64_t k, int slot_shift, HsLocal& L, const RepTab& R) {
    uint32_t slot = (uint32_t)(k >> slot_shift) & (HS_SLOTS - 1);
    for (int probes = 0; probes < HS_SLOTS; ++probes) {
        unsigned long long cur = *reinterpret_cast<volatile unsigned long long*>(&tab[slot]);
        if (cur == EMPTY64) {
            cur = atomicCAS(&tab[slot], EMPTY64, (unsigned long long)k);
            if (cur == EMPTY64) {
                ++L.distinct;
                return;
            }
        }
        if (cur == k) {
            const uint32_t bit = 1u << (slot & 31);
            if (!(*reinterpret_cast<volatile uint32_t*>(&twice[slot >> 5]) & bit)) {
                const uint32_t prev = atomicOr(&twice[slot >> 5], bit);
                if (!(prev & bit)) {
                    ++L.dups;
                    if (MASK) rep_insert64(R, fmix64_inv(k));
                }
            }
            return;
        }
        slot = (slot + 1) & (HS_SLOTS - 1);
    }
    L.overflow = 1;
}

// H (buffer ctl->result of k0 / k1): n hashes sorted by their low bits (h & mask). slot_shift: first hash bit above the mask.
template <bool MASK>
__global__ void __launch_bounds__(HS_THREADS) hs_dedup_kernel(const uint64_t* __restrict__ k0, const uint64_t* __restrict__ k1, const RsControl* ctl,
                                                              int64_t n, uint64_t mask, int slot_shift, HsCounters* ctr, RepTab R) {
    extern __shared__ __align__(16) uint8_t hs_smem[];
    unsigned long long* tab = reinterpret_cast<unsigned long long*>(hs_smem);
    uint32_t* twice = reinterpret_cast<uint32_t*>(hs_smem + (size_t)HS_SLOTS * 8);
    const uint64_t* __restrict__ H = ctl->result ? k1 : k0;
    const int tid = threadIdx.x;
    HsLocal L{0, 0, 0};
    uint32_t skew = 0;
    const int64_t n_chunks = (n + HS_CHUNK - 1) / HS_CHUNK;
    for (int64_t chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
        for (int i = tid; i < HS_SLOTS; i += HS_THREADS) tab[i] = EMPTY64;
        for (int i = tid; i < HS_SLOTS / 32; i += HS_THREADS) twice[i] = 0u;
        __syncthreads();
        const int64_t s = chunk * HS_CHUNK, e = s + HS_CHUNK < n ? s + HS_CHUNK : n;
        const bool has_prev = s > 0;
        const uint64_t b_prev = has_prev ? (__ldg(H + s - 1) & mask) : 0ull;  // the bucket that may reach into this chunk: its owner's
        const uint64_t b_last = __ldg(H + e - 1) & mask;
        {
            uint64_t kb[HS_CHUNK / HS_THREADS];  // (all loads of the chunk in flight together)
#pragma unroll
            for (int i = 0; i < HS_CHUNK / HS_THREADS; ++i) {
                const int64_t j = s + i * HS_THREADS + tid;
                kb[i] = j < e ? __ldg(H + j) : b_prev;
            }
#pragma unroll
            for (int i = 0; i < HS_CHUNK / HS_THREADS; ++i) {
                const int64_t j = s + i * HS_THREADS + tid;
                if (j < e && (!has_prev || (kb[i] & mask) != b_prev)) hs_insert<MASK>(tab, twice, kb[i], slot_shift, L, R);
            }
        }
        // the chunk's last bucket, if it began inside the chunk, is ours to its end. The first HS_SPEC rounds past the chunk
        // are loaded at once without waiting for the round before (sorted input: a key beyond the bucket fails the compare)
        if (e < n && (!has_prev || b_last != b_prev)) {
            uint64_t kk[HS_SPEC];
#pragma unroll
            for (int r = 0; r < HS_SPEC; ++r) {
                const int64_t j = e + (int64_t)r * HS_THREADS + tid;
                kk[r] = j < n ? __ldg(H + j) : ~b_last;  // (~b_last & mask != b_last)
            }
#pragma unroll
            for (int r = 0; r < HS_SPEC; ++r)
                if ((kk[r] & mask) == b_last) hs_insert<MASK>(tab, twice, kk[r], slot_shift, L, R);
            for (int r = HS_SPEC;; ++r) {
                const int64_t jl = e + (int64_t)r * HS_THREADS - 1;  // (sorted: the last key of the round before decides for all)
                if (jl >= n || (__ldg(H + jl) & mask) != b_last) break;
                if (r >= HS_MAX_TAIL_ROUNDS) {
                    skew = 1;
                    break;
                }
                const int64_t j = e + (int64_t)r * HS_THREADS + tid;
                if (j < n) {
                    const uint64_t k = __ldg(H + j);
                    if ((k & mask) == b_last) hs_insert<MASK>(tab, twice, k, slot_shift, L, R);
                }
            }
        }
        __syncthreads();
    }
    flush_counter_block((unsigned long long)L.distinct, &ctr->distinct);
    flush_counter_block((unsigned long long)L.dups, &ctr->dup_keys);
    flush_counter_block((unsigned long long)L.overflow, &ctr->overflow);
    flush_counter_block((unsigned long long)skew, &ctr->skew);
}

bool distinct64_sorted(Engine& e, const Column& c, int64_t n, Distinct64Result& r, int& launches, const RepTab* R) {
    if (n <= 0 || n >= ((int64_t)1 << 30) || getenv("TG_HASH_NO_SORTED")) return false;
    if (R) rep_reset(e, *R);
    int n_passes = n > ((int64_t)1 << 27) ? 3 : 2;
    if (const char* f = getenv("TG_HS_PASSES")) n_passes = atoi(f) == 3 ? 3 : n_passes;  // (tests reach the 24-bit bucket mode without 2^27 rows)
    const size_t keys_b = hs_round_up((size_t)n * 8, 256), tmp_b = hs_round_up(rs_temp_bytes(n, n_passes), 256);
    uint8_t* scr = e.scratch(2 * keys_b + tmp_b + 256);
    uint64_t* bufs[2] = {(uint64_t*)scr, (uint64_t*)(scr + keys_b)};
    uint8_t* temp = scr + 2 * keys_b;
    HsCounters* d_ctr = (HsCounters*)(scr + 2 * keys_b + tmp_b);
    TG_CUDA(cudaMemsetAsync(d_ctr, 0, sizeof(HsCounters), e.stream));
    const RsTemp T0 = rs_temp_carve(temp, n, n_passes);  // (ctl / hist / base sit at fixed offsets: the same for any n)
    TG_CUDA(cudaMemsetAsync(T0.hist, 0, (size_t)RS_MAX_PASSES * RS_BINS * 8, e.stream));
    const int64_t n_tiles = (n + HS_TILE - 1) / HS_TILE;
    const int pgrid = (int)std::max<int64_t>(1, std::min<int64_t>(n_tiles, (int64_t)e.sm_count * 4));
    hs_prep_kernel<<<pgrid, HS_THREADS, 0, e.stream>>>((const uint64_t*)c.values.p, (const uint32_t*)c.validity.p, n, c.dtype == TG_FLOAT64, bufs[0], d_ctr,
                                                         T0.hist, n_passes);
    TG_CUDA(cudaGetLastError());
    ++launches;
    HsCounters h{};
    TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    const int64_t nv = (int64_t)h.n_valid;
    if (nv > 0) {
        const RsTemp T = rs_temp_carve(temp, nv, n_passes);
        uint32_t* no_vals[2] = {nullptr, nullptr};
        launches += rs_sort_pairs<uint32_t>(e.stream, bufs, no_vals, nv, 0, n_passes, false, T, e.sm_count, nullptr, true);
        const size_t smem = (size_t)HS_SLOTS * 8 + HS_SLOTS / 8;
        auto* dedup = R ? hs_dedup_kernel<true> : hs_dedup_kernel<false>;
        TG_CUDA(cudaFuncSetAttribute(dedup, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int64_t n_chunks = (nv + HS_CHUNK - 1) / HS_CHUNK;
        int per_sm = 1;
        TG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, dedup, HS_THREADS, smem));
        const int dgrid = (int)std::max<int64_t>(1, std::min<int64_t>(n_chunks, (int64_t)e.sm_count * std::max(per_sm, 1)));
        dedup<<<dgrid, HS_THREADS, smem, e.stream>>>(bufs[0], bufs[1], T.ctl, nv, ((uint64_t)1 << (8 * n_passes)) - 1, 8 * n_passes, d_ctr,
                                                     R ? *R : RepTab{});
        TG_CUDA(cudaGetLastError());
        ++launches;
        TG_CUDA(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, e.stream));
        TG_CUDA(cudaStreamSynchronize(e.stream));
        if (h.overflow || h.skew) return false;
    }
    // the key whose hash is the EMPTY word is counted apart (R holds keys: its key is an ordinary one there)
    if (R && h.special > 1) rep_mark(e, *R, fmix64_inv(EMPTY64));
    r.distinct = h.distinct + (h.special ? 1 : 0);
    r.dup_keys = h.dup_keys + (h.special > 1 ? 1 : 0);
    r.nulls = h.nulls;
    return true;
}

}  // namespace tg
