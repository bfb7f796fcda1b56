// K2 — string pattern kernel: host-compiled byte DFAs run over Arrow Utf8 (offsets + value bytes).
//
// Replaces `COUNT(CASE WHEN [TRIM(]c[)] ~|~* 'pat' ... THEN 1 END), COUNT(*)`
// (constraints/format.rs:762-776 -> arrow-string regexp_is_match -> regex crate) for every pattern that a
// suite applies to the same column, in ONE pass over that column's bytes.
//
// Host: the DFAs of all patterns on a column (regex_dfa.cpp) are combined into ONE product automaton over a
// joint byte-class map, so an input byte costs one class lookup and one transition lookup however many
// patterns are checked. Product states whose components are all decided (DEAD = cannot match any more,
// MATCH = already matched) are numbered first, so "nothing left to learn from this string" is a single
// compare. The built-in formats are anchored (^...$) and die within a few bytes on strings of another
// format, which keeps the product small (the C3 suite '@' + email + SSN + credit card: 669 states x 82
// classes); when a product would not fit in shared memory the patterns are split into several passes.
//
// Device: warp-per-32-strings, thread-per-string. A warp owns blocks of 32 consecutive rows, whose bytes are
// one contiguous range of the value buffer: lane 0 fetches that range with one TMA bulk copy
// (cp.async.bulk -> mbarrier) into the warp's private double buffer one block ahead, and the offsets two
// blocks ahead, so the DFA loop only ever touches shared memory (bytes, class map, transition table).
// A block whose bytes exceed the warp's stage (very long strings) is walked straight from global memory.
#include <algorithm>
#include <cstring>
#include <map>
#include <mutex>

#include "engine.hpp"
#include "ptx.cuh"
#include "regex_dfa.hpp"

namespace tg {

constexpr int STR_MAX_DFA = 8;          // patterns per product automaton
constexpr int STR_MAX_WARPS = 32;       // warps per CTA (upper bound; fewer when the table is large)
constexpr size_t STR_SMEM_MAX = 227 * 1024 - 2048;   // dynamic shared memory available beside the static tables
constexpr size_t STR_TABLE_BUDGET = 112 * 1024;      // product tables up to this size still leave room for 32 warps
constexpr size_t STR_SINGLE_BUDGET = 200 * 1024;     // a single pattern may take this much (fewer warps per CTA then)
constexpr uint32_t STR_MAX_ELEMS = 131072 - 512;     // transition entries addressable by the 16-bit row encoding (rows start at even elements)

// Transition table encoding (all uint16). A product state is named by HALF THE ELEMENT INDEX of its row (rows are padded
// to an even number of entries, so 16 bits name rows of tables up to 256 KB — more than shared memory holds; the big
// automata are the ones with Unicode word boundaries). A row has n_classes entries (next state per joint byte class)
// plus one END entry: the match mask if the string ends in this state. Decided states (every component DEAD or MATCH)
// come first, so "decided" is E < n_term * stride / 2;
// their rows loop to themselves. Byte 0xFF — which cannot occur in valid UTF-8 — is a class of its own that maps
// every state to itself: the kernel pads the last 8-byte window of a string with 0xFF, so the per-byte loop has no
// end-of-string test and no branch at all; "decided" is tested once per 8 bytes.
struct StrParams {
    const int32_t* offsets;
    const uint8_t* bytes;
    const uint32_t* validity;
    int64_t n_rows;
    int64_t n_blocks;         // ceil(n_rows / 32)
    int32_t trim;             // TRIM(c) (ASCII space, both ends) before matching
    uint32_t n_classes;       // joint byte classes
    uint32_t term_limit;      // states with E < term_limit are decided
    uint32_t start;           // encoded start state
    uint32_t tab_bytes;       // 256-byte class map + transition table (multiple of 16)
    uint32_t stage;           // bytes per warp stage buffer (multiple of 128)
    const uint8_t* g_blob;    // [256 B class map (uint8 class)][table]
    unsigned long long* out;  // [STR_MAX_DFA] match counts, [STR_MAX_DFA] = valid (non-null) rows
    uint32_t* bits[STR_MAX_DFA];  // MASK kernels: per pattern, one match word per 32 rows of the table (null: not requested)
};

extern __shared__ __align__(256) uint8_t str_smem[];

__device__ __forceinline__ uint32_t lds_u8(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// 8 automaton steps over the bytes of (lo, hi). cls_base = shared address of the class map (256-byte aligned, so
// "base + byte" is one PRMT); the 8 class lookups do not depend on the state and issue ahead of the chain.
// DIRECT: the table's rows are indexed by the BYTE itself (small automata: rows of 256 + END entries fit shared memory), so a
// byte costs ONE shared load instead of two — the kernel is bound by the shared-memory pipe.
template <bool DIRECT>
__device__ __forceinline__ uint32_t dfa_step8(uint32_t lo, uint32_t hi, uint32_t E, uint32_t cls_base, uint32_t tab_addr) {
    uint32_t c[8];
    if constexpr (DIRECT) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            c[k] = (lo >> (8 * k)) & 255u;
            c[4 + k] = (hi >> (8 * k)) & 255u;
        }
    } else {
        c[0] = lds_u8(__byte_perm(lo, cls_base, 0x7650));
        c[1] = lds_u8(__byte_perm(lo, cls_base, 0x7651));
        c[2] = lds_u8(__byte_perm(lo, cls_base, 0x7652));
        c[3] = lds_u8(__byte_perm(lo, cls_base, 0x7653));
        c[4] = lds_u8(__byte_perm(hi, cls_base, 0x7650));
        c[5] = lds_u8(__byte_perm(hi, cls_base, 0x7651));
        c[6] = lds_u8(__byte_perm(hi, cls_base, 0x7652));
        c[7] = lds_u8(__byte_perm(hi, cls_base, 0x7653));
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) E = lds_u16(tab_addr + 2u * (2u * E + c[k]));
    return E;
}

// Runs the product automaton over bytes [p, e) of the warp's stage (shared address stage_addr).
template <bool DIRECT>
__device__ __forceinline__ uint32_t run_dfa_smem(uint32_t stage_addr, uint32_t p, uint32_t e, uint32_t E, uint32_t cls_base,
                                                 uint32_t tab_addr, uint32_t term_limit) {
    while (p < e) {
        const uint32_t a = stage_addr + (p & ~3u);
        const uint32_t w0 = lds_u32(a), w1 = lds_u32(a + 4), w2 = lds_u32(a + 8);
        const uint32_t sh = (p & 3u) * 8u;
        uint32_t lo = __funnelshift_r(w0, w1, sh), hi = __funnelshift_r(w1, w2, sh);
        const uint32_t rem = e - p;
        if (rem < 8u) {  // pad the tail with 0xFF (the identity class)
            const unsigned long long m = ~0ull << (8u * rem);
            lo |= (uint32_t)m;
            hi |= (uint32_t)(m >> 32);
        }
        E = dfa_step8<DIRECT>(lo, hi, E, cls_base, tab_addr);
        p += 8u;
        if (E < term_limit) break;
    }
    return E;
}
// Same over global memory, byte loads (only blocks whose bytes exceed the stage: very long strings).
template <bool DIRECT>
__device__ __forceinline__ uint32_t run_dfa_gmem(const uint8_t* bytes, uint32_t p, uint32_t e, uint32_t E, uint32_t cls_base,
                                                 uint32_t tab_addr, uint32_t term_limit) {
    for (; p < e && E >= term_limit; ++p) {
        const uint32_t b = __ldg(bytes + p);
        E = lds_u16(tab_addr + 2u * (2u * E + (DIRECT ? b : lds_u8(cls_base + b))));
    }
    return E;
}

// R = rows per lane per block: a warp's block is 32*R consecutive rows (lane l owns rows base + j*32 + l, j < R).
// R = 2 halves the per-block bookkeeping (offset prefetch, TMA issue, mbarrier wait) per string and evens out the
// string-length imbalance between lanes; R = 1 keeps small inputs spread over all SMs.
// MASK: also store, per requested pattern, the word of every 32 rows whose bit l says "row of lane l matched"
template <int NDFA, int R, bool DIRECT, bool MASK>
__global__ void __launch_bounds__(STR_MAX_WARPS * 32) dfa_kernel(const __grid_constant__ StrParams P) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    // ---- stage class map + transition table ----
    {
        const uint4* src = reinterpret_cast<const uint4*>(P.g_blob);
        uint4* dst = reinterpret_cast<uint4*>(str_smem);
        for (uint32_t i = threadIdx.x; i < P.tab_bytes / 16; i += blockDim.x) dst[i] = src[i];
    }
    const uint32_t cls_base = smem_u32(str_smem), tab_addr = cls_base + 256u;
    const uint32_t term_limit = P.term_limit, n_classes = P.n_classes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(str_smem + P.tab_bytes) + warp * 2;
    const uint32_t stage_bytes = P.stage;
    uint8_t* stage = str_smem + P.tab_bytes + (size_t)n_warps * 16 + (size_t)warp * (2 * stage_bytes);
    const uint32_t stage_addr = smem_u32(stage);
    if (lane == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
    }
    mbar_fence_init();
    __syncthreads();

    const int64_t total_warps = (int64_t)gridDim.x * n_warps;
    const int64_t gwarp = (int64_t)blockIdx.x * n_warps + warp;
    const int64_t n = P.n_rows;
    uint32_t cnt[NDFA];
#pragma unroll
    for (int i = 0; i < NDFA; ++i) cnt[i] = 0;
    uint32_t nvalid = 0;
    const uint32_t byte_base_lo = (uint32_t)reinterpret_cast<uint64_t>(P.bytes) & 15u;  // misalignment of the value buffer

    // a block's per-lane view: [o, oe) of its R rows (rows past the end are empty) and their validity words
    struct Blk {
        uint32_t o[R], oe[R], vw[R];
    };
    auto load_offsets = [&](int64_t blk, Blk& b) {
#pragma unroll
        for (int j = 0; j < R; ++j) {
            b.o[j] = b.oe[j] = 0;
            b.vw[j] = 0;
        }
        if (blk < P.n_blocks) {
#pragma unroll
            for (int j = 0; j < R; ++j) {
                const int64_t r = (blk * R + j) * 32 + lane;
                b.o[j] = (uint32_t)__ldg(P.offsets + (r < n ? r : n));
                b.oe[j] = (uint32_t)__ldg(P.offsets + (r + 1 < n ? r + 1 : n));
                b.vw[j] = ((blk * R + j) * 32 < n) ? (P.validity ? __ldg(P.validity + blk * R + j) : 0xffffffffu) : 0u;
            }
        }
    };
    // block byte range -> TMA bulk copy into stage buffer `buf`. Returns false when the block is empty or does not
    // fit (then it is read from global memory); org = the byte index (relative to P.bytes, may be "negative" by the
    // buffer's misalignment, hence wrapping uint32 arithmetic) that maps to stage offset 0. 16 bytes of the stage
    // stay free: the window loads of the last string may run 11 bytes past its end.
    auto issue = [&](const Blk& b, int buf, uint32_t& org) -> bool {
        const uint32_t b0 = __shfl_sync(0xffffffffu, b.o[0], 0), b1 = __shfl_sync(0xffffffffu, b.oe[R - 1], 31);
        if (b1 <= b0) return false;
        const uint32_t lead = (byte_base_lo + b0) & 15u;  // bytes between the 16-byte aligned start and b0
        const uint32_t sz = (lead + (b1 - b0) + 15u) & ~15u;
        if (sz + 16u > stage_bytes) return false;
        if (lane == 0) {
            mbar_arrive_expect_tx(&bars[buf], sz);
            bulk_g2s(stage + buf * stage_bytes, P.bytes + (int64_t)b0 - (int64_t)lead, sz, &bars[buf]);
        }
        org = b0 - lead;
        return true;
    };

    Blk c0, c1, c2;  // blocks it, it+1, it+2
    load_offsets(gwarp, c0);
    load_offsets(gwarp + total_warps, c1);
    uint32_t org0 = 0, org1 = 0;  // stage origins of blocks it, it+1
    bool staged0 = false, staged1 = false;
    if (gwarp < P.n_blocks) staged0 = issue(c0, 0, org0);
    uint32_t phase = 0;  // bit b = parity of the next completion of bars[b]
    int it = 0;
    for (int64_t blk = gwarp; blk < P.n_blocks; blk += total_warps, ++it) {
        const int buf = it & 1;
        // prefetch: offsets two blocks ahead, bytes one block ahead (its buffer was last read an iteration ago)
        load_offsets(blk + 2 * total_warps, c2);
        __syncwarp();
        staged1 = false;
        if (blk + total_warps < P.n_blocks) staged1 = issue(c1, buf ^ 1, org1);
        // ---- this block ----
        if (staged0) {
            mbar_wait(&bars[buf], (phase >> buf) & 1u);
            phase ^= 1u << buf;
        }
#pragma unroll
        for (int j = 0; j < R; ++j) {
            const bool valid = (c0.vw[j] >> lane) & 1u;
            uint32_t m = 0;
            if (valid && (blk * R + j) * 32 + lane < n) {
                ++nvalid;
                uint32_t E;
                if (staged0) {
                    uint32_t p = c0.o[j] - org0, e = c0.oe[j] - org0;
                    if (P.trim) {
                        const uint8_t* base = stage + buf * stage_bytes;
                        while (p < e && base[p] == ' ') ++p;
                        while (e > p && base[e - 1] == ' ') --e;
                    }
                    E = run_dfa_smem<DIRECT>(stage_addr + buf * stage_bytes, p, e, P.start, cls_base, tab_addr, term_limit);
                } else {
                    uint32_t p = c0.o[j], e = c0.oe[j];
                    if (P.trim) {
                        while (p < e && P.bytes[p] == ' ') ++p;
                        while (e > p && P.bytes[e - 1] == ' ') --e;
                    }
                    E = run_dfa_gmem<DIRECT>(P.bytes, p, e, P.start, cls_base, tab_addr, term_limit);
                }
                m = lds_u16(tab_addr + 2u * (2u * E + n_classes));  // END entry = match mask
#pragma unroll
                for (int i = 0; i < NDFA; ++i) cnt[i] += (m >> i) & 1u;
            }
            if constexpr (MASK) {
                // every lane of the warp is here (the block loop is warp-uniform); NULL rows and rows past the end match nothing
#pragma unroll
                for (int i = 0; i < NDFA; ++i)
                    if (P.bits[i]) {
                        const uint32_t w = __ballot_sync(0xffffffffu, (m >> i) & 1u);
                        if (lane == 0 && (blk * R + j) * 32 < n) P.bits[i][blk * R + j] = w;
                    }
            }
        }
        c0 = c1;
        c1 = c2;
        org0 = org1;
        staged0 = staged1;
    }
    // ---- block reduction -> one atomic per counter per CTA ----
    __syncthreads();
    uint32_t* red = reinterpret_cast<uint32_t*>(str_smem + P.tab_bytes + (size_t)n_warps * 16);  // stages are dead now
#pragma unroll
    for (int i = 0; i <= NDFA; ++i) {
        uint32_t v = i < NDFA ? cnt[i < NDFA ? i : 0] : nvalid;
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
        if (lane == 0) red[i * STR_MAX_WARPS + warp] = v;
    }
    __syncthreads();
    if (threadIdx.x <= NDFA) {
        unsigned long long v = 0;
        for (int k = 0; k < n_warps; ++k) v += red[threadIdx.x * STR_MAX_WARPS + k];
        if (v) atomicAdd(P.out + (threadIdx.x < NDFA ? threadIdx.x : STR_MAX_DFA), v);
    }
}

static size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ------------------------------------------------------------------ product automaton (host) ----
struct Product {
    uint32_t n_classes = 0, n_states = 0, n_term = 0, term_limit = 0, start = 0, tab_bytes = 0;
    std::vector<uint8_t> blob;  // device image, see StrParams::g_blob
    bool ok = false;            // false: exceeded the state / size limits
    bool direct = false;        // rows indexed by the byte (n_classes == 256): dfa_kernel<.., DIRECT = true>
};

static Product build_product(const std::vector<const Dfa*>& dfas, size_t table_budget, bool allow_direct) {
    Product pr;
    const size_t nd = dfas.size();
    // joint byte classes
    std::map<std::vector<uint8_t>, uint16_t> sig_ids;
    uint16_t jclass[256];
    std::vector<uint8_t> rep;
    for (int b = 0; b < 256; ++b) {
        std::vector<uint8_t> sig;
        for (auto* d : dfas) sig.push_back(d->class_of[b]);
        sig.push_back(b == 0xFF ? 1 : 0);  // 0xFF (never part of valid UTF-8) is the kernel's padding byte: own class
        auto it = sig_ids.find(sig);
        if (it == sig_ids.end()) {
            it = sig_ids.emplace(sig, (uint16_t)rep.size()).first;
            rep.push_back((uint8_t)b);
        }
        jclass[b] = it->second;
    }
    const uint32_t njc = (uint32_t)rep.size(), stride = (njc + 2) & ~1u, nop_class = jclass[0xFF];  // njc entries + END, padded to even
    if (njc > 255) return pr;
    // breadth-first product construction
    typedef std::vector<uint16_t> Tuple;
    std::map<Tuple, uint32_t> ids;
    std::vector<Tuple> states;
    std::vector<uint32_t> next;  // [state][class] in discovery numbering
    Tuple st0;
    for (auto* d : dfas) st0.push_back((uint16_t)d->start);
    ids[st0] = 0;
    states.push_back(st0);
    const size_t max_elems = std::min<size_t>(STR_MAX_ELEMS, table_budget / 2);
    const size_t max_states = max_elems / stride;
    for (size_t s = 0; s < states.size(); ++s) {
        for (uint32_t c = 0; c < njc; ++c) {
            Tuple t(nd);
            const Tuple& cur = states[s];
            if (c == nop_class) {
                t = cur;  // identity: the padding byte
            } else {
                for (size_t i = 0; i < nd; ++i) {
                    uint16_t x = cur[i];
                    if (x > DFA_MATCH) x = dfas[i]->next[(size_t)x * dfas[i]->n_classes + dfas[i]->class_of[rep[c]]];
                    t[i] = x;
                }
            }
            auto it = ids.find(t);
            if (it == ids.end()) {
                if (states.size() >= max_states) return pr;
                it = ids.emplace(t, (uint32_t)states.size()).first;
                states.push_back(std::move(t));
            }
            next.push_back(it->second);
        }
    }
    const uint32_t ns = (uint32_t)states.size();
    // rows: decided tuples (every component DEAD or MATCH) first
    std::vector<uint32_t> enc(ns);
    uint32_t n_term = 0;
    auto decided = [&](const Tuple& t) {
        for (auto x : t)
            if (x > DFA_MATCH) return false;
        return true;
    };
    for (uint32_t s = 0; s < ns; ++s)
        if (decided(states[s])) enc[s] = (n_term++) * (stride / 2);
    uint32_t row = n_term;
    for (uint32_t s = 0; s < ns; ++s)
        if (!decided(states[s])) enc[s] = (row++) * (stride / 2);
    if ((size_t)ns * stride > max_elems) return pr;
    // small automata: rows indexed by the byte itself (256 entries + END, padded to 258), when that table still fits the budget
    // (and the 16-bit row names: E = row * 129)
    if (allow_direct && (size_t)ns * 258 * 2 + 256 <= table_budget && (size_t)ns * 129 < 65536) {
        const uint32_t dstride = 258;
        uint32_t nt = 0;
        for (uint32_t s = 0; s < ns; ++s)
            if (decided(states[s])) enc[s] = (nt++) * (dstride / 2);
        uint32_t drow = nt;
        for (uint32_t s = 0; s < ns; ++s)
            if (!decided(states[s])) enc[s] = (drow++) * (dstride / 2);
        const size_t tb = round_up(256 + (size_t)ns * dstride * 2, 16);
        pr.n_classes = 256;
        pr.n_states = ns;
        pr.n_term = nt;
        pr.term_limit = nt * (dstride / 2);
        pr.start = enc[0];
        pr.tab_bytes = (uint32_t)tb;
        pr.blob.assign(tb, 0);
        for (int b = 0; b < 256; ++b) pr.blob[b] = (uint8_t)jclass[b];  // (unused by the direct kernel)
        uint16_t* dtab = reinterpret_cast<uint16_t*>(pr.blob.data() + 256);
        for (uint32_t s = 0; s < ns; ++s) {
            uint8_t m = 0;
            for (size_t i = 0; i < nd; ++i) {
                const uint16_t x = states[s][i];
                if (x == DFA_MATCH || (x != DFA_DEAD && dfas[i]->accept_end[x])) m |= (uint8_t)(1u << i);
            }
            uint16_t* r = dtab + 2 * (size_t)enc[s];
            for (int b = 0; b < 256; ++b) r[b] = (uint16_t)enc[next[(size_t)s * njc + jclass[b]]];
            r[256] = m;  // END entry (index n_classes)
        }
        pr.direct = true;
        pr.ok = true;
        return pr;
    }
    const size_t tab_bytes = round_up(256 + (size_t)ns * stride * 2, 16);
    pr.n_classes = njc;
    pr.n_states = ns;
    pr.n_term = n_term;
    pr.term_limit = n_term * (stride / 2);
    pr.start = enc[0];
    pr.tab_bytes = (uint32_t)tab_bytes;
    pr.blob.assign(tab_bytes, 0);
    for (int b = 0; b < 256; ++b) pr.blob[b] = (uint8_t)jclass[b];
    uint16_t* tab = reinterpret_cast<uint16_t*>(pr.blob.data() + 256);
    for (uint32_t s = 0; s < ns; ++s) {
        uint8_t m = 0;
        for (size_t i = 0; i < nd; ++i) {
            const uint16_t x = states[s][i];
            if (x == DFA_MATCH || (x != DFA_DEAD && dfas[i]->accept_end[x])) m |= (uint8_t)(1u << i);
        }
        uint16_t* r = tab + 2 * (size_t)enc[s];
        for (uint32_t c = 0; c < njc; ++c) r[c] = (uint16_t)enc[next[(size_t)s * njc + c]];
        r[njc] = m;  // END entry
    }
    pr.ok = true;
    return pr;
}

// products are cached by their pattern list, like the reference caches compiled patterns (format.rs:183-184)
static const Product& cached_product(const std::vector<std::pair<std::string, bool>>& pats, size_t budget) {
    static std::mutex mu;
    static std::map<std::pair<std::vector<std::pair<std::string, bool>>, size_t>, Product> cache;
    std::lock_guard<std::mutex> g(mu);
    const bool allow_direct = getenv("TG_STR_NO_DIRECT") == nullptr;  // (tests run both table layouts against the oracle)
    auto key = std::make_pair(pats, budget * 2 + (allow_direct ? 1 : 0));
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    std::vector<Dfa> dfas;
    for (auto& p : pats) dfas.push_back(compile_regex(p.first, p.second));
    std::vector<const Dfa*> ptrs;
    for (auto& d : dfas) ptrs.push_back(&d);
    return cache.emplace(key, build_product(ptrs, budget, allow_direct)).first->second;
}

typedef void (*Kernel)(const StrParams);
template <bool MASK>
static Kernel pick_dfa_kernel(int nd, int R, bool direct) {
    const Kernel k1 = nd <= 1 ? (Kernel)dfa_kernel<1, 1, false, MASK> : nd <= 2 ? (Kernel)dfa_kernel<2, 1, false, MASK> : nd <= 4 ? (Kernel)dfa_kernel<4, 1, false, MASK> : (Kernel)dfa_kernel<8, 1, false, MASK>;
    const Kernel k2 = nd <= 1 ? (Kernel)dfa_kernel<1, 2, false, MASK> : nd <= 2 ? (Kernel)dfa_kernel<2, 2, false, MASK> : nd <= 4 ? (Kernel)dfa_kernel<4, 2, false, MASK> : (Kernel)dfa_kernel<8, 2, false, MASK>;
    const Kernel d1 = nd <= 1 ? (Kernel)dfa_kernel<1, 1, true, MASK> : nd <= 2 ? (Kernel)dfa_kernel<2, 1, true, MASK> : nd <= 4 ? (Kernel)dfa_kernel<4, 1, true, MASK> : (Kernel)dfa_kernel<8, 1, true, MASK>;
    const Kernel d2 = nd <= 1 ? (Kernel)dfa_kernel<1, 2, true, MASK> : nd <= 2 ? (Kernel)dfa_kernel<2, 2, true, MASK> : nd <= 4 ? (Kernel)dfa_kernel<4, 2, true, MASK> : (Kernel)dfa_kernel<8, 2, true, MASK>;
    return direct ? (R == 2 ? d2 : d1) : (R == 2 ? k2 : k1);
}

static void run_string_pass(Engine& e, Table& t, Plan& p, Column& c, const std::vector<int>& ids, const Product& pr, bool trim) {
    const int nd = (int)ids.size();
    StrParams P{};
    bool masks = false;
    for (int i = 0; i < nd; ++i) {
        P.bits[i] = p.aggs[ids[i]].bits;
        masks |= P.bits[i] != nullptr;
    }
    P.trim = trim ? 1 : 0;
    P.n_classes = pr.n_classes;
    P.term_limit = pr.term_limit;
    P.start = pr.start;
    P.tab_bytes = pr.tab_bytes;
    // per-warp stage: 32 rows of ~1.5x the column's mean length, so almost every block is staged by TMA
    const double mean_len = t.n_rows > 0 ? (double)c.value_bytes / (double)t.n_rows : 0.0;
    // two rows per lane once there are enough 64-row blocks to keep every warp of the grid busy several times over
    static const int64_t r2_min_rows = [] {
        const char* ev = getenv("TG_STR_R2_MIN_ROWS");  // tests lower it so both block shapes meet the oracle
        const long long x = ev ? atoll(ev) : 0;
        return x > 0 ? (int64_t)x : (int64_t)1 << 21;
    }();
    const int R = t.n_rows >= r2_min_rows && !getenv("TG_STR_R1") ? 2 : 1;
    size_t stage = round_up((size_t)(mean_len * 32.0 * R * (R == 2 ? 1.25 : 1.5)) + (R == 2 ? 128 : 256), 128);
    stage = std::min<size_t>(std::max<size_t>(stage, 1024), 8192);
    // warps per CTA: as many as fit beside the table (each owns a double stage + 2 mbarriers)
    int warps = 0;
    for (;; stage = std::max<size_t>(1024, stage / 2 / 128 * 128)) {
        warps = (int)std::min<size_t>(STR_MAX_WARPS, (STR_SMEM_MAX - pr.tab_bytes) / (2 * stage + 16));
        if (warps >= 8 || stage <= 1024) break;
    }
    if (warps < 1) throw Error(TG_ERR_UNSUPPORTED, "DFA tables exceed shared memory");
    P.stage = (uint32_t)stage;
    const size_t smem = pr.tab_bytes + (size_t)warps * (2 * stage + 16);
    const size_t blob_bytes = round_up(pr.blob.size(), 256);
    uint8_t* scr = e.scratch(blob_bytes + 256);
    TG_CUDA(cudaMemcpyAsync(scr, pr.blob.data(), pr.blob.size(), cudaMemcpyHostToDevice, e.stream));
    unsigned long long* d_out = reinterpret_cast<unsigned long long*>(scr + blob_bytes);
    TG_CUDA(cudaMemsetAsync(d_out, 0, 128, e.stream));
    P.g_blob = scr;
    P.out = d_out;
    P.offsets = reinterpret_cast<const int32_t*>(c.offsets.p);
    P.bytes = c.values.p;
    P.validity = reinterpret_cast<const uint32_t*>(c.validity.p);
    P.n_rows = t.n_rows;
    P.n_blocks = (t.n_rows + 32 * R - 1) / (32 * R);
    const Kernel kernel = masks ? pick_dfa_kernel<true>(nd, R, pr.direct) : pick_dfa_kernel<false>(nd, R, pr.direct);
    TG_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)STR_SMEM_MAX));
    const int threads = warps * 32;
    int per_sm = 1;
    TG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    per_sm = std::max(per_sm, 1);
    const int64_t ctas_needed = (P.n_blocks + warps - 1) / warps;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(ctas_needed, (int64_t)e.sm_count * per_sm));
    TG_CUDA(cudaEventRecord(e.ev[2], e.stream));
    kernel<<<grid, threads, smem, e.stream>>>(P);
    TG_CUDA(cudaGetLastError());
    TG_CUDA(cudaEventRecord(e.ev[3], e.stream));
    e.launches += 1;
    p.stats.launches += 1;
    unsigned long long h_out[16];
    TG_CUDA(cudaMemcpyAsync(h_out, d_out, 128, cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    float ms = 0;
    TG_CUDA(cudaEventElapsedTime(&ms, e.ev[2], e.ev[3]));
    p.stats.string_ms += ms;
    p.stats.gpu_ms += ms;
    for (int i = 0; i < nd; ++i) {
        Agg& a = p.aggs[ids[i]];
        a.u[0] = h_out[i];
        a.u[1] = (uint64_t)t.n_rows - h_out[STR_MAX_DFA];
        a.u[2] = (uint64_t)t.n_rows;
    }
}

void exec_string_jobs(Engine& e, Table& t, Plan& p, const std::vector<int>& agg_ids) {
    // group by (column, TRIM flag): all patterns of a group walk the same byte sequence, so they share one
    // product automaton (split greedily when the product would not fit in shared memory)
    std::map<std::pair<Column*, bool>, std::vector<int>> by_col;
    std::vector<Column*> counted;
    for (int id : agg_ids) {
        Agg& a = p.aggs[id];
        Column* c = t.find(a.cols[0]);
        if (!c) {
            a.err = TG_ERR_COLUMN_NOT_FOUND;
            a.err_msg = "Schema error: No field named " + a.cols[0] + ". Valid fields are " + t.valid_fields() + ".";
            continue;
        }
        if (c->dtype != TG_UTF8) {
            a.err = TG_ERR_TYPE_MISMATCH;
            a.err_msg = "Error during planning: regular expression match requires a Utf8 column, '" + c->name + "' is not";
            continue;
        }
        by_col[{c, (a.flags & 2) != 0}].push_back(id);
        if (std::find(counted.begin(), counted.end(), c) == counted.end()) {
            counted.push_back(c);
            // algorithmic bytes: offsets + value bytes + validity, once per column
            p.stats.bytes_scanned += (uint64_t)(t.n_rows + 1) * 4 + (uint64_t)c->value_bytes +
                                     (c->validity.p ? (uint64_t)(t.n_rows + 7) / 8 : 0);
        }
    }
    for (auto& kv : by_col) {
        Column& c = *kv.first.first;
        const bool trim = kv.first.second;
        if (t.n_rows == 0) {
            for (int id : kv.second) p.aggs[id].u[2] = 0;
            continue;
        }
        std::vector<int> pass;
        std::vector<std::pair<std::string, bool>> pats;
        auto flush = [&]() {
            if (pass.empty()) return;
            const Product* pr = &cached_product(pats, STR_TABLE_BUDGET);
            if (!pr->ok && pass.size() == 1) pr = &cached_product(pats, STR_SINGLE_BUDGET);  // alone it may take most of shared memory
            if (!pr->ok) {
                for (int id : pass) {
                    p.aggs[id].err = TG_ERR_UNSUPPORTED;
                    p.aggs[id].err_msg = "regex pattern compiles to DFA tables that exceed shared memory";
                }
            } else {
                run_string_pass(e, t, p, c, pass, *pr, trim);
            }
            pass.clear();
            pats.clear();
        };
        for (int id : kv.second) {
            const std::pair<std::string, bool> pat{p.aggs[id].text, (p.aggs[id].flags & 1) != 0};
            if (!pass.empty()) {
                auto trial = pats;
                trial.push_back(pat);
                if (pass.size() >= (size_t)STR_MAX_DFA || !cached_product(trial, STR_TABLE_BUDGET).ok) flush();
            }
            pass.push_back(id);
            pats.push_back(pat);
        }
        flush();
    }
}

// ------------------------------------------------------------------ LENGTH(c) ranges ----
// Replaces COUNT(CASE WHEN LENGTH(c) >= a [AND LENGTH(c) <= b] OR c IS NULL THEN 1 END) * 1.0 / NULLIF(COUNT(*), 0)
// (constraints/length.rs:150-170) for every length assertion on a column in one pass. SQL LENGTH counts CHARACTERS:
// bytes minus UTF-8 continuation bytes. A row's byte length (two offsets) already bounds its character count
// (ceil(bytes/4) <= chars <= bytes), so the value bytes are only read for rows some range cannot decide from that.
constexpr int LEN_MAX_RANGES = 8;

// SQL LENGTH of one non-null row: bytes minus the UTF-8 continuation bytes (need_bytes false: the byte count, unused then)
template <class LP>
__device__ __forceinline__ long long row_chars(const LP& P, int32_t b, int32_t e, bool need_bytes, uint64_t w0, uint64_t w1) {
    if (!need_bytes) return e - b;
    int cont = __popcll(w0 & (~w0 << 1) & 0x8080808080808080ull) + __popcll(w1 & (~w1 << 1) & 0x8080808080808080ull);
    for (int32_t q = b + 16; q < e; q += 8) {
        const uint64_t w = load_upto8(P.bytes, q, min(8, e - q));
        cont += __popcll(w & (~w << 1) & 0x8080808080808080ull);
    }
    return (long long)(e - b) - cont;
}
constexpr int LEN_THREADS = 256;
constexpr int LEN_ILP = 4;
struct LenParams {
    const int32_t* offsets;
    const uint8_t* bytes;
    const uint32_t* validity;
    int64_t n_rows;
    int32_t n_ranges;
    int32_t pad;
    long long lo[LEN_MAX_RANGES], hi[LEN_MAX_RANGES];
    unsigned long long* out;  // [LEN_MAX_RANGES] matching non-null rows, [LEN_MAX_RANGES] = non-null rows
    uint32_t* bits[LEN_MAX_RANGES];  // MASK kernel: per requested range, one word per 32 rows (bit set: non-null and in range)
};

template <bool MASK>
__global__ void __launch_bounds__(LEN_THREADS) length_kernel(const __grid_constant__ LenParams P) {
    uint32_t cnt[LEN_MAX_RANGES];
#pragma unroll
    for (int i = 0; i < LEN_MAX_RANGES; ++i) cnt[i] = 0;
    uint32_t nvalid = 0;
    for (int64_t base = (int64_t)blockIdx.x * LEN_THREADS * LEN_ILP; base < P.n_rows; base += (int64_t)gridDim.x * LEN_THREADS * LEN_ILP) {
        int32_t b[LEN_ILP], e[LEN_ILP];
        uint32_t vw[LEN_ILP];
#pragma unroll
        for (int k = 0; k < LEN_ILP; ++k) {
            const int64_t row = base + (int64_t)k * LEN_THREADS + threadIdx.x;
            const int64_t rc = row < P.n_rows ? row : P.n_rows - 1;
            b[k] = __ldg(P.offsets + rc);
            e[k] = __ldg(P.offsets + rc + 1);
            vw[k] = P.validity ? __ldg(P.validity + (rc >> 5)) : 0xffffffffu;
        }
        // wave 2: which rows need their bytes, and the first 16 bytes of those (all loads before any counting)
        bool live[LEN_ILP], need[LEN_ILP];
        uint64_t w0[LEN_ILP], w1[LEN_ILP];
#pragma unroll
        for (int k = 0; k < LEN_ILP; ++k) {
            const int64_t row = base + (int64_t)k * LEN_THREADS + threadIdx.x;
            live[k] = row < P.n_rows && ((vw[k] >> (row & 31)) & 1u);
            const long long nbytes = e[k] - b[k], min_chars = (nbytes + 3) >> 2;
            need[k] = false;
            for (int i = 0; i < P.n_ranges; ++i) {
                const bool surely_out = nbytes < P.lo[i] || min_chars > P.hi[i];
                const bool surely_in = min_chars >= P.lo[i] && nbytes <= P.hi[i];
                need[k] |= !(surely_out || surely_in);
            }
            need[k] = need[k] && live[k];
            w0[k] = need[k] && nbytes > 0 ? load_upto8(P.bytes, b[k], (int)(nbytes < 8 ? nbytes : 8)) : 0ull;
            w1[k] = need[k] && nbytes > 8 ? load_upto8(P.bytes, b[k] + 8, (int)(nbytes - 8 < 8 ? nbytes - 8 : 8)) : 0ull;
        }
#pragma unroll
        for (int k = 0; k < LEN_ILP; ++k) {
            if constexpr (MASK) {
                // the ballot needs every lane: NULL rows and rows past the end are out of every range
                uint32_t inm = 0;
                if (live[k]) {
                    ++nvalid;
                    const long long chars = row_chars(P, b[k], e[k], need[k], w0[k], w1[k]);
                    const long long nbytes = e[k] - b[k], min_chars = (nbytes + 3) >> 2;
#pragma unroll
                    for (int i = 0; i < LEN_MAX_RANGES; ++i)
                        if (i < P.n_ranges) {
                            const bool in = need[k] ? (chars >= P.lo[i] && chars <= P.hi[i]) : (min_chars >= P.lo[i] && nbytes <= P.hi[i]);
                            cnt[i] += in;
                            inm |= (uint32_t)in << i;
                        }
                }
                const int64_t row = base + (int64_t)k * LEN_THREADS + threadIdx.x;
#pragma unroll
                for (int i = 0; i < LEN_MAX_RANGES; ++i)
                    if (i < P.n_ranges && P.bits[i]) {
                        const uint32_t w = __ballot_sync(0xffffffffu, (inm >> i) & 1u);
                        if ((threadIdx.x & 31) == 0 && row < P.n_rows) P.bits[i][row >> 5] = w;
                    }
                continue;
            }
            if (!live[k]) continue;
            ++nvalid;
            const long long nbytes = e[k] - b[k], min_chars = (nbytes + 3) >> 2;
            const bool need_bytes = need[k];
            long long chars = nbytes;
            if (need_bytes) {
                // 10xxxxxx bytes are UTF-8 continuation bytes: not characters
                int cont = __popcll(w0[k] & (~w0[k] << 1) & 0x8080808080808080ull) + __popcll(w1[k] & (~w1[k] << 1) & 0x8080808080808080ull);
                for (int32_t q = b[k] + 16; q < e[k]; q += 8) {
                    const uint64_t w = load_upto8(P.bytes, q, min(8, e[k] - q));
                    cont += __popcll(w & (~w << 1) & 0x8080808080808080ull);
                }
                chars = nbytes - cont;
            }
#pragma unroll
            for (int i = 0; i < LEN_MAX_RANGES; ++i)
                if (i < P.n_ranges) {
                    // when the bytes were skipped every range was decided from the bounds alone
                    const bool in = need_bytes ? (chars >= P.lo[i] && chars <= P.hi[i]) : (min_chars >= P.lo[i] && nbytes <= P.hi[i]);
                    cnt[i] += in;
                }
        }
    }
    __shared__ unsigned long long red[LEN_MAX_RANGES + 1][LEN_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i <= LEN_MAX_RANGES; ++i) {
        uint32_t v = i < LEN_MAX_RANGES ? cnt[i < LEN_MAX_RANGES ? i : 0] : nvalid;
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
        if (lane == 0) red[i][warp] = v;
    }
    __syncthreads();
    if (threadIdx.x <= LEN_MAX_RANGES) {
        unsigned long long v = 0;
        for (int k = 0; k < LEN_THREADS / 32; ++k) v += red[threadIdx.x][k];
        if (v) atomicAdd(P.out + threadIdx.x, v);
    }
}

void exec_length_jobs(Engine& e, Table& t, Plan& p, const std::vector<int>& agg_ids) {
    std::map<Column*, std::vector<int>> by_col;
    for (int id : agg_ids) {
        Agg& a = p.aggs[id];
        Column* c = t.find(a.cols[0]);
        if (!c) {
            a.err = TG_ERR_COLUMN_NOT_FOUND;
            a.err_msg = "Schema error: No field named " + a.cols[0] + ". Valid fields are " + t.valid_fields() + ".";
            continue;
        }
        if (c->dtype != TG_UTF8) {
            a.err = TG_ERR_TYPE_MISMATCH;
            a.err_msg = "Error during planning: LENGTH requires a Utf8 column, '" + c->name + "' is not";
            continue;
        }
        by_col[c].push_back(id);
    }
    for (auto& kv : by_col) {
        Column& c = *kv.first;
        p.stats.bytes_scanned += (uint64_t)(t.n_rows + 1) * 4 + (uint64_t)c.value_bytes + (c.validity.p ? (uint64_t)(t.n_rows + 7) / 8 : 0);
        for (size_t first = 0; first < kv.second.size(); first += LEN_MAX_RANGES) {
            const size_t cnt = std::min<size_t>(LEN_MAX_RANGES, kv.second.size() - first);
            unsigned long long h_out[16] = {0};
            if (t.n_rows > 0) {
                LenParams P{};
                P.offsets = reinterpret_cast<const int32_t*>(c.offsets.p);
                P.bytes = c.values.p;
                P.validity = reinterpret_cast<const uint32_t*>(c.validity.p);
                P.n_rows = t.n_rows;
                P.n_ranges = (int)cnt;
                for (size_t i = 0; i < cnt; ++i) {
                    P.lo[i] = p.aggs[kv.second[first + i]].lo;
                    P.hi[i] = p.aggs[kv.second[first + i]].hi;
                }
                uint8_t* scr = e.scratch(256);
                P.out = reinterpret_cast<unsigned long long*>(scr);
                TG_CUDA(cudaMemsetAsync(scr, 0, 128, e.stream));
                const int64_t per_cta = (int64_t)LEN_THREADS * LEN_ILP;
                const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((t.n_rows + per_cta - 1) / per_cta, (int64_t)e.sm_count * 8));
                bool masks = false;
                for (size_t i = 0; i < cnt; ++i) {
                    P.bits[i] = p.aggs[kv.second[first + i]].bits;
                    masks |= P.bits[i] != nullptr;
                }
                TG_CUDA(cudaEventRecord(e.ev[2], e.stream));
                if (masks) length_kernel<true><<<grid, LEN_THREADS, 0, e.stream>>>(P);
                else length_kernel<false><<<grid, LEN_THREADS, 0, e.stream>>>(P);
                TG_CUDA(cudaGetLastError());
                TG_CUDA(cudaEventRecord(e.ev[3], e.stream));
                TG_CUDA(cudaMemcpyAsync(h_out, scr, 128, cudaMemcpyDeviceToHost, e.stream));
                TG_CUDA(cudaStreamSynchronize(e.stream));
                float ms = 0;
                TG_CUDA(cudaEventElapsedTime(&ms, e.ev[2], e.ev[3]));
                p.stats.string_ms += ms;
                p.stats.gpu_ms += ms;
                p.stats.launches += 1;
                e.launches += 1;
            }
            for (size_t i = 0; i < cnt; ++i) {
                Agg& a = p.aggs[kv.second[first + i]];
                a.u[0] = h_out[i];
                a.u[1] = (uint64_t)t.n_rows - h_out[LEN_MAX_RANGES];
                a.u[2] = (uint64_t)t.n_rows;
            }
        }
    }
}

}  // namespace tg
