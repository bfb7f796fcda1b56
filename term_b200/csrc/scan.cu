// K1 — fused single-pass numeric scan (sm_100a).
//
// Replaces, for a whole suite at once, the per-constraint DataFusion aggregates
//   COUNT(*) / COUNT(c)            constraints/completeness.rs:158, analyzers/basic/completeness.rs:106
//   MIN/MAX/AVG/SUM/STDDEV/VARIANCE constraints/statistics.rs:263, analyzers/basic/{mean,min_max,sum}.rs
//   CORR / COVAR_SAMP / raw co-sums constraints/correlation.rs:313, analyzers/advanced/correlation.rs:239
//   COUNT(CASE WHEN pred THEN 1 END) constraints/custom_sql.rs:203, analyzers/advanced/compliance.rs:153
//
// Design (B200-first, HBM-bound):
//   * persistent CTAs, one per SM; each CTA walks row tiles round-robin.
//   * warp 0 is a TMA producer: for every tile it issues one cp.async.bulk (UBLKCP) per referenced
//     buffer (values and validity words of each column) into a multi-stage shared-memory ring,
//     completion tracked by mbarrier transaction bytes. Every input byte crosses HBM->SM exactly once
//     no matter how many constraints reference it.
//   * 16 consumer warps each own "units" (one aggregate over a row slice of the tile, a multiple of 128
//     rows); they read the tile from shared memory conflict-free (lane-contiguous 8-byte elements) and
//     release the stage through an "empty" mbarrier, so fast warps run up to n_stages-1 tiles ahead of
//     slow ones. When a pass has at most 16 units (the planner replicates aggregates over row slices to
//     get exactly 16) every warp keeps its unit's descriptor and accumulators in REGISTERS for the whole
//     scan; with more units a warp runs several per tile against per-lane state in shared memory.
//   * descriptor tables (columns, units, predicate code) are copied to shared memory once; every
//     kind / flag decision is hoisted out of the row loops (template specialisations).
//   * every inner loop handles 128 rows per iteration (4 groups of 32 rows; lane l owns row 32g+l) with
//     ONE 128-bit load of the four validity words and two independent accumulator sets, so each dependent
//     FP64 chain has a second one to overlap with.
//   * moments are accumulated as shifted sums Σ(x-K), Σ(x-K)² with K a typical element of the column; NULL
//     rows are masked by zeroing the shifted value (2 selects) or by AND-ing the validity predicate into the
//     compare (min/max, predicates: no extra instruction).
//   * per-CTA partials go to global memory; scan_finalize_kernel reduces them in a fixed order, so a
//     given (grid, plan) is bit-reproducible run to run.
#include <cfloat>
#include <cstddef>
#include <cstdio>
#include <math_constants.h>

#include "ptx.cuh"
#include "scan_defs.h"

namespace tg {

extern __shared__ __align__(128) uint8_t scan_smem[];

typedef uint64_t Slots[SCAN_STATE_SLOTS];

__device__ __forceinline__ uint32_t tail_mask(int base_row, int rows_in_tile) {
    const int rem = rows_in_tile - base_row;
    return rem >= 32 ? 0xffffffffu : (rem <= 0 ? 0u : ((1u << rem) - 1u));
}
__device__ __forceinline__ double u2d(uint64_t u) { return __longlong_as_double((long long)u); }
__device__ __forceinline__ uint64_t d2u(double d) { return (uint64_t)__double_as_longlong(d); }

// validity word (32 rows) of a column inside the stage; all-ones when the column has no bitmap
__device__ __forceinline__ uint32_t vword(const ScanColDesc& c, const uint8_t* stage, int word) {
    return c.validity ? reinterpret_cast<const uint32_t*>(stage + c.smem_bits_off)[word] : 0xffffffffu;
}
__device__ __forceinline__ uint32_t word_or_ones(const uint32_t* bits, bool has_bits, int g) { return has_bits ? bits[g] : 0xffffffffu; }

// masked running min / max: the validity predicate is AND-ed into the compare (DSETP.x.AND / ISETP.x.AND.EX), so
// masking costs no extra instruction
__device__ __forceinline__ void min_if_f64(double& mn, double x, uint32_t m) {
    asm("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %2, 0;\n\tsetp.lt.and.f64 q, %1, %0, p;\n\tselp.f64 %0, %1, %0, q;\n\t}" : "+d"(mn) : "d"(x), "r"(m));
}
__device__ __forceinline__ void max_if_f64(double& mx, double x, uint32_t m) {
    asm("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %2, 0;\n\tsetp.gt.and.f64 q, %1, %0, p;\n\tselp.f64 %0, %1, %0, q;\n\t}" : "+d"(mx) : "d"(x), "r"(m));
}
__device__ __forceinline__ void min_if_i64(int64_t& mn, int64_t x, uint32_t m) {
    asm("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %2, 0;\n\tsetp.lt.and.s64 q, %1, %0, p;\n\tselp.b64 %0, %1, %0, q;\n\t}" : "+l"(mn) : "l"(x), "r"(m));
}
__device__ __forceinline__ void max_if_i64(int64_t& mx, int64_t x, uint32_t m) {
    asm("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %2, 0;\n\tsetp.gt.and.s64 q, %1, %0, p;\n\tselp.b64 %0, %1, %0, q;\n\t}" : "+l"(mx) : "l"(x), "r"(m));
}

// ======================================================================================================
// Units. Every unit kind is a small object: setup(descriptors) / load(slots) / tile(stage) / store(slots).
// `slots` is this lane's SCAN_STATE_SLOTS 64-bit partial state (meaning per kind in scan_defs.h).
// The last (partial) tile of the table takes a generic masked path (`tail`).
// ======================================================================================================

// ---- COUNT: popcount of validity words ----
struct CountUnit {
    static constexpr bool MASK = false;
    uint32_t bits_off;
    int w0, nw, row0, lane;
    uint64_t n;
    __device__ __forceinline__ void setup(const ScanTables& T, const ScanUnitDesc& u, int lane_) {
        const ScanColDesc& c = T.cols[u.c0];
        bits_off = c.validity ? c.smem_bits_off : 0xffffffffu;
        w0 = u.row0 >> 5;
        nw = u.nrows >> 5;
        row0 = u.row0;
        lane = lane_;
    }
    __device__ __forceinline__ void load(const Slots& r) { n = r[S_N]; }
    __device__ __forceinline__ void tile(const uint8_t* stage, int rows, bool partial) {
        if (bits_off == 0xffffffffu && !partial) {
            if (lane == 0) n += (uint64_t)nw * 32;
            return;
        }
        for (int j = lane; j < nw; j += 32) {
            uint32_t w = bits_off != 0xffffffffu ? reinterpret_cast<const uint32_t*>(stage + bits_off)[w0 + j] : 0xffffffffu;
            if (partial) w &= tail_mask(row0 + 32 * j, rows);
            n += __popc(w);
        }
    }
    __device__ __forceinline__ void store(Slots& r) {
#pragma unroll
        for (int k = 0; k < SCAN_STATE_SLOTS; ++k) r[k] = 0;
        r[S_N] = n;
    }
};

// ---- NUM: n, Σ(x-K), Σ(x-K)², min, max, wrapping integer sum over the valid rows of one column ----
template <bool IS_I64, int FLAGS>
struct NumUnit {
    static constexpr bool MOM = (FLAGS & UF_MOMENTS) != 0, MM = (FLAGS & UF_MINMAX) != 0, ISUM = IS_I64 && (FLAGS & UF_ISUM) != 0;
    static constexpr bool MASK = false;
    uint32_t val_off, bits_off;  // bits_off == ~0u: no bitmap
    int row0, nrows, lane;
    double K;
    uint64_t n, isum[2];
    double sd[2], sdd[2], fmn[2], fmx[2];
    int64_t imn[2], imx[2];

    __device__ __forceinline__ void setup(const ScanTables& T, const ScanUnitDesc& u, int lane_) {
        const ScanColDesc& c = T.cols[u.c0];
        val_off = c.smem_val_off;
        bits_off = c.validity ? c.smem_bits_off : 0xffffffffu;
        row0 = u.row0;
        nrows = u.nrows;
        lane = lane_;
        K = c.pivot;
    }
    __device__ __forceinline__ void load(const Slots& r) {
        n = r[S_N];
        sd[0] = u2d(r[S_SD]);
        sdd[0] = u2d(r[S_SDD]);
        fmn[0] = u2d(r[S_MIN]);
        fmx[0] = u2d(r[S_MAX]);
        imn[0] = (int64_t)r[S_MIN];
        imx[0] = (int64_t)r[S_MAX];
        isum[0] = r[S_ISUM];
        sd[1] = sdd[1] = 0.0;
        fmn[1] = CUDART_INF;
        fmx[1] = -CUDART_INF;
        imn[1] = INT64_MAX;
        imx[1] = INT64_MIN;
        isum[1] = 0;
    }
    // m != 0 <=> the row is valid; MASKED = false: every row is valid (m ignored)
    template <int A, bool MASKED>
    __device__ __forceinline__ void acc(uint64_t raw, uint32_t m) {
        if (IS_I64) {
            const int64_t xi = (int64_t)raw;
            if (MOM) {
                double d = (double)xi - K;
                if (MASKED) d = m ? d : 0.0;
                sd[A] += d;
                sdd[A] = fma(d, d, sdd[A]);
            }
            if (ISUM) isum[A] += (MASKED && !m) ? 0ull : raw;
            if (MM) {
                if (MASKED) {
                    min_if_i64(imn[A], xi, m);
                    max_if_i64(imx[A], xi, m);
                } else {
                    imn[A] = xi < imn[A] ? xi : imn[A];
                    imx[A] = xi > imx[A] ? xi : imx[A];
                }
            }
        } else {
            const double x = u2d(raw);
            if (MOM) {
                double d = x - K;
                if (MASKED) d = m ? d : 0.0;
                sd[A] += d;
                sdd[A] = fma(d, d, sdd[A]);
            }
            if (MM) {
                if (MASKED) {
                    min_if_f64(fmn[A], x, m);
                    max_if_f64(fmx[A], x, m);
                } else {
                    fmn[A] = x < fmn[A] ? x : fmn[A];
                    fmx[A] = x > fmx[A] ? x : fmx[A];
                }
            }
        }
    }
    template <bool HB>
    __device__ __forceinline__ void body(const uint8_t* stage) {
        const uint64_t* vals = reinterpret_cast<const uint64_t*>(stage + val_off) + row0 + lane;
        const uint32_t lanebit = 1u << lane;
        const int nq = nrows >> 7;
        if (HB) {
            const uint32_t* bits = reinterpret_cast<const uint32_t*>(stage + bits_off) + (row0 >> 5);
            for (int j = lane; j < 4 * nq; j += 32) n += __popc(bits[j]);
            if (FLAGS == 0) return;
            const uint4* b4 = reinterpret_cast<const uint4*>(bits);
#pragma unroll 2
            for (int q = 0; q < nq; ++q) {
                const uint4 w = b4[q];
                const uint64_t r0 = vals[128 * q], r1 = vals[128 * q + 32], r2 = vals[128 * q + 64], r3 = vals[128 * q + 96];
                acc<0, true>(r0, w.x & lanebit);
                acc<1, true>(r1, w.y & lanebit);
                acc<0, true>(r2, w.z & lanebit);
                acc<1, true>(r3, w.w & lanebit);
            }
        } else {
            if (lane == 0) n += (uint64_t)nrows;
            if (FLAGS == 0) return;
#pragma unroll 2
            for (int q = 0; q < nq; ++q) {
                const uint64_t r0 = vals[128 * q], r1 = vals[128 * q + 32], r2 = vals[128 * q + 64], r3 = vals[128 * q + 96];
                acc<0, false>(r0, 1u);
                acc<1, false>(r1, 1u);
                acc<0, false>(r2, 1u);
                acc<1, false>(r3, 1u);
            }
        }
    }
    // last tile of the table: rows beyond `rows` are masked off
    __device__ __forceinline__ void tail(const uint8_t* stage, int rows) {
        const uint64_t* vals = reinterpret_cast<const uint64_t*>(stage + val_off) + row0 + lane;
        const bool has_bits = bits_off != 0xffffffffu;
        const uint32_t* bits = reinterpret_cast<const uint32_t*>(stage + (has_bits ? bits_off : 0u)) + (row0 >> 5);
        const int ng = nrows >> 5;
        for (int j = lane; j < ng; j += 32) n += __popc(word_or_ones(bits, has_bits, j) & tail_mask(row0 + 32 * j, rows));
        if (FLAGS == 0) return;
#pragma unroll 1
        for (int g = 0; g < ng; ++g) {
            const uint32_t w = word_or_ones(bits, has_bits, g) & tail_mask(row0 + 32 * g, rows);
            acc<0, true>(vals[32 * g], (w >> lane) & 1u);
        }
    }
    __device__ __forceinline__ void tile(const uint8_t* stage, int rows, bool partial) {
        if (partial) tail(stage, rows);
        else if (bits_off != 0xffffffffu) body<true>(stage);
        else body<false>(stage);
    }
    __device__ __forceinline__ void store(Slots& r) {
#pragma unroll
        for (int k = 0; k < SCAN_STATE_SLOTS; ++k) r[k] = 0;
        r[S_N] = n;
        r[S_SD] = d2u(sd[0] + sd[1]);
        r[S_SDD] = d2u(sdd[0] + sdd[1]);
        if (IS_I64) {
            r[S_MIN] = (uint64_t)(imn[0] < imn[1] ? imn[0] : imn[1]);
            r[S_MAX] = (uint64_t)(imx[0] > imx[1] ? imx[0] : imx[1]);
        } else {
            r[S_MIN] = d2u(fmn[0] < fmn[1] ? fmn[0] : fmn[1]);
            r[S_MAX] = d2u(fmx[0] > fmx[1] ? fmx[0] : fmx[1]);
        }
        r[S_ISUM] = isum[0] + isum[1];
    }
};

// ---- PAIR: co-moments over the rows where both columns are valid ----
template <bool XI, bool YI>
struct PairUnit {
    static constexpr bool MASK = false;
    uint32_t vx_off, vy_off, bx_off, by_off;
    int row0, nrows, lane;
    double Kx, Ky, sx[2], sy[2], sxx[2], syy[2], sxy[2];
    uint64_t n;
    __device__ __forceinline__ void setup(const ScanTables& T, const ScanUnitDesc& u, int lane_) {
        const ScanColDesc& cx = T.cols[u.c0];
        const ScanColDesc& cy = T.cols[u.c1];
        vx_off = cx.smem_val_off;
        vy_off = cy.smem_val_off;
        bx_off = cx.validity ? cx.smem_bits_off : 0xffffffffu;
        by_off = cy.validity ? cy.smem_bits_off : 0xffffffffu;
        row0 = u.row0;
        nrows = u.nrows;
        lane = lane_;
        Kx = cx.pivot;
        Ky = cy.pivot;
    }
    __device__ __forceinline__ void load(const Slots& r) {
        n = r[P_N];
        sx[0] = u2d(r[P_SX]);
        sy[0] = u2d(r[P_SY]);
        sxx[0] = u2d(r[P_SXX]);
        syy[0] = u2d(r[P_SYY]);
        sxy[0] = u2d(r[P_SXY]);
        sx[1] = sy[1] = sxx[1] = syy[1] = sxy[1] = 0.0;
    }
    template <int A, bool MASKED>
    __device__ __forceinline__ void acc(uint64_t rx, uint64_t ry, uint32_t m) {
        double dx = (XI ? (double)(int64_t)rx : u2d(rx)) - Kx;
        double dy = (YI ? (double)(int64_t)ry : u2d(ry)) - Ky;
        if (MASKED) {
            dx = m ? dx : 0.0;
            dy = m ? dy : 0.0;
        }
        sx[A] += dx;
        sy[A] += dy;
        sxx[A] = fma(dx, dx, sxx[A]);
        syy[A] = fma(dy, dy, syy[A]);
        sxy[A] = fma(dx, dy, sxy[A]);
    }
    template <int NB>  // number of bitmaps: 0, 1 (at b1_off) or 2
    __device__ __forceinline__ void body(const uint8_t* stage, uint32_t b1_off, uint32_t b2_off) {
        const uint64_t* vx = reinterpret_cast<const uint64_t*>(stage + vx_off) + row0 + lane;
        const uint64_t* vy = reinterpret_cast<const uint64_t*>(stage + vy_off) + row0 + lane;
        const uint32_t lanebit = 1u << lane;
        const int nq = nrows >> 7;
        const uint32_t* bits1 = reinterpret_cast<const uint32_t*>(stage + (NB ? b1_off : 0u)) + (row0 >> 5);
        const uint32_t* bits2 = reinterpret_cast<const uint32_t*>(stage + (NB == 2 ? b2_off : 0u)) + (row0 >> 5);
        if (NB) {
            for (int j = lane; j < 4 * nq; j += 32) n += __popc(NB == 2 ? (bits1[j] & bits2[j]) : bits1[j]);
        } else if (lane == 0) {
            n += (uint64_t)nrows;
        }
        const uint4* p1 = reinterpret_cast<const uint4*>(bits1);
        const uint4* p2 = reinterpret_cast<const uint4*>(bits2);
#pragma unroll 2
        for (int q = 0; q < nq; ++q) {
            uint4 w = make_uint4(lanebit, lanebit, lanebit, lanebit);
            if (NB >= 1) w = p1[q];
            if (NB == 2) {
                const uint4 w2 = p2[q];
                w.x &= w2.x;
                w.y &= w2.y;
                w.z &= w2.z;
                w.w &= w2.w;
            }
            const uint64_t x0 = vx[128 * q], x1 = vx[128 * q + 32], x2 = vx[128 * q + 64], x3 = vx[128 * q + 96];
            const uint64_t y0 = vy[128 * q], y1 = vy[128 * q + 32], y2 = vy[128 * q + 64], y3 = vy[128 * q + 96];
            acc<0, NB != 0>(x0, y0, w.x & lanebit);
            acc<1, NB != 0>(x1, y1, w.y & lanebit);
            acc<0, NB != 0>(x2, y2, w.z & lanebit);
            acc<1, NB != 0>(x3, y3, w.w & lanebit);
        }
    }
    __device__ __forceinline__ uint32_t both(const uint8_t* stage, int word) const {
        uint32_t w = 0xffffffffu;
        if (bx_off != 0xffffffffu) w &= reinterpret_cast<const uint32_t*>(stage + bx_off)[word];
        if (by_off != 0xffffffffu) w &= reinterpret_cast<const uint32_t*>(stage + by_off)[word];
        return w;
    }
    __device__ __forceinline__ void tail(const uint8_t* stage, int rows) {
        const uint64_t* vx = reinterpret_cast<const uint64_t*>(stage + vx_off) + row0 + lane;
        const uint64_t* vy = reinterpret_cast<const uint64_t*>(stage + vy_off) + row0 + lane;
        const int ng = nrows >> 5, w0 = row0 >> 5;
        for (int j = lane; j < ng; j += 32) n += __popc(both(stage, w0 + j) & tail_mask(row0 + 32 * j, rows));
#pragma unroll 1
        for (int g = 0; g < ng; ++g) {
            const uint32_t w = both(stage, w0 + g) & tail_mask(row0 + 32 * g, rows);
            acc<0, true>(vx[32 * g], vy[32 * g], (w >> lane) & 1u);
        }
    }
    __device__ __forceinline__ void tile(const uint8_t* stage, int rows, bool partial) {
        const bool hx = bx_off != 0xffffffffu, hy = by_off != 0xffffffffu;
        if (partial) tail(stage, rows);
        else if (hx && hy) body<2>(stage, bx_off, by_off);
        else if (hx || hy) body<1>(stage, hx ? bx_off : by_off, 0u);
        else body<0>(stage, 0u, 0u);
    }
    __device__ __forceinline__ void store(Slots& r) {
#pragma unroll
        for (int k = 0; k < SCAN_STATE_SLOTS; ++k) r[k] = 0;
        r[P_N] = n;
        r[P_SX] = d2u(sx[0] + sx[1]);
        r[P_SY] = d2u(sy[0] + sy[1]);
        r[P_SXX] = d2u(sxx[0] + sxx[1]);
        r[P_SYY] = d2u(syy[0] + syy[1]);
        r[P_SXY] = d2u(sxy[0] + sxy[1]);
    }
};

// ---- TERMS: AND / OR of <= 4 comparison terms ----
// Term-major over blocks of up to 32 row groups: one pass per term leaves, in every lane, a 32-bit mask whose bit g
// says "term is TRUE for MY row of group g" (row 32g + lane); the validity bit is AND-ed into the compare as a
// predicate. Masks of the terms are AND-ed / OR-ed and popcounted per lane: no cross-lane traffic at all, and
// the (kind, operator) dispatch happens once per term per block, outside the row loop.
template <int KIND, int OP, bool HB>  // OP = cmp_mask: 1 <, 2 ==, 3 <=, 4 >, 5 <> (13 with unordered), 6 >=
__device__ __forceinline__ uint32_t term_loop(uint64_t imm, const uint64_t* vals, const uint4* b4, int nq, uint32_t lanebit) {
    uint32_t pm = 0;
#pragma unroll 2
    for (int q = 0; q < nq; ++q) {
        uint4 w = make_uint4(lanebit, lanebit, lanebit, lanebit);
        if (HB) w = b4[q];
        const uint64_t raw[4] = {vals[128 * q], vals[128 * q + 32], vals[128 * q + 64], vals[128 * q + 96]};
        const uint32_t v[4] = {w.x & lanebit, w.y & lanebit, w.z & lanebit, w.w & lanebit};
        uint32_t nib = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            bool r;
            if (KIND == TK_I64) {
                const int64_t x = (int64_t)raw[j], c = (int64_t)imm;
                r = OP == 1 ? x < c : OP == 2 ? x == c : OP == 3 ? x <= c : OP == 4 ? x > c : OP == 6 ? x >= c : x != c;
            } else {
                // floats: NaN sorts above every number (Arrow total order): > and >= and <> are true for NaN
                const double x = KIND == TK_F64 ? u2d(raw[j]) : (double)(int64_t)raw[j], c = u2d(imm);
                r = OP == 1 ? x < c : OP == 2 ? x == c : OP == 3 ? x <= c : OP == 4 ? !(x <= c) : OP == 6 ? !(x < c) : x != c;
            }
            if (r && (!HB || v[j])) nib |= 1u << j;
        }
        pm |= nib << (4 * q);
    }
    return pm;
}
template <int KIND, bool HB>
__device__ __forceinline__ uint32_t term_ops(int cmp_mask, uint64_t imm, const uint64_t* vals, const uint4* b4, int nq, uint32_t lanebit) {
    switch (cmp_mask & 7) {
        case 1: return term_loop<KIND, 1, HB>(imm, vals, b4, nq, lanebit);
        case 2: return term_loop<KIND, 2, HB>(imm, vals, b4, nq, lanebit);
        case 3: return term_loop<KIND, 3, HB>(imm, vals, b4, nq, lanebit);
        case 4: return term_loop<KIND, 4, HB>(imm, vals, b4, nq, lanebit);
        case 6: return term_loop<KIND, 6, HB>(imm, vals, b4, nq, lanebit);
        default: return term_loop<KIND, 5, HB>(imm, vals, b4, nq, lanebit);
    }
}
// validity of MY rows of a block: bit g = row (32 g + lane) is valid
__device__ __forceinline__ uint32_t valid_loop(const uint4* b4, int nq, uint32_t lanebit) {
    uint32_t pm = 0;
    for (int q = 0; q < nq; ++q) {
        const uint4 w = b4[q];
        const uint32_t nib = ((w.x & lanebit) ? 1u : 0u) | ((w.y & lanebit) ? 2u : 0u) | ((w.z & lanebit) ? 4u : 0u) | ((w.w & lanebit) ? 8u : 0u);
        pm |= nib << (4 * q);
    }
    return pm;
}

// MASK_: also store the TRUE word of every 32 rows to the aggregate's bit buffer (tile_row0 = the tile's first table row)
template <bool MASK_>
struct TermsUnit {
    static constexpr bool MASK = MASK_;
    const ScanTables* T;
    int t0, nt, row0, nrows, lane;
    bool is_or;
    uint64_t cnt;
    uint32_t *bits, *tbits;  // the aggregate's words / those of the current tile (null: no verdicts requested)
    __device__ __forceinline__ void at_tile(int64_t tile_row0) { tbits = bits ? bits + (tile_row0 >> 5) : nullptr; }
    __device__ __forceinline__ void setup(const ScanTables& T_, const ScanUnitDesc& u, int lane_) {
        if constexpr (MASK) bits = u.bits;
        T = &T_;
        t0 = u.code_off;
        nt = u.code_len;
        row0 = u.row0;
        nrows = u.nrows;
        lane = lane_;
        is_or = u.flags & 1;
    }
    __device__ __forceinline__ void load(const Slots& r) { cnt = r[0]; }
    __device__ __forceinline__ void tile(const uint8_t* stage, int rows, bool partial) {
        const uint32_t lanebit = 1u << lane;
        for (int blk = 0; blk < nrows; blk += 1024) {
            const int base = row0 + blk;
            const int nq = min(8, (nrows - blk) >> 7);
            uint32_t m = is_or ? 0u : 0xffffffffu;
#pragma unroll 1
            for (int k = 0; k < nt; ++k) {
                // term descriptors are read from shared memory once per (term, block): a few uniform loads
                const ScanTerm& t = T->terms[t0 + k];
                const ScanColDesc& c = T->cols[t.col];
                const bool hb = c.validity != nullptr;
                const int kind = t.kind, cmp = t.cmp_mask;
                const uint64_t imm = t.imm;
                const uint64_t* vals = reinterpret_cast<const uint64_t*>(stage + c.smem_val_off) + base + lane;
                const uint4* b4 = reinterpret_cast<const uint4*>(stage + (hb ? c.smem_bits_off : 0u) + (base >> 3));
                uint32_t pm;
                if (kind == TK_ISNULL || kind == TK_NOTNULL) {
                    pm = hb ? valid_loop(b4, nq, lanebit) : 0xffffffffu;
                    if (kind == TK_ISNULL) pm = ~pm;
                } else if (kind == TK_F64) {
                    pm = hb ? term_ops<TK_F64, true>(cmp, imm, vals, b4, nq, lanebit) : term_ops<TK_F64, false>(cmp, imm, vals, b4, nq, lanebit);
                } else if (kind == TK_I64) {
                    pm = hb ? term_ops<TK_I64, true>(cmp, imm, vals, b4, nq, lanebit) : term_ops<TK_I64, false>(cmp, imm, vals, b4, nq, lanebit);
                } else {
                    pm = hb ? term_ops<TK_I64_AS_F64, true>(cmp, imm, vals, b4, nq, lanebit)
                            : term_ops<TK_I64_AS_F64, false>(cmp, imm, vals, b4, nq, lanebit);
                }
                m = is_or ? (m | pm) : (m & pm);
            }
            // keep the groups of this block whose row (base + 32 g + lane) exists
            int ng = 4 * nq;
            if (partial) ng = max(0, min(ng, (rows - base - lane + 31) >> 5));
            const uint32_t gmask = ng >= 32 ? 0xffffffffu : ((1u << ng) - 1u);
            cnt += __popc(m & gmask);
            if (MASK && tbits) {
                // transpose: lane g collects the word of group g (bit l = row base + 32 g + l); a 32-row word lies in exactly
                // one unit slice of one tile, so it has exactly one writer
                const int ngrp = 4 * nq;
                uint32_t word = 0;
                for (int g = 0; g < ngrp; ++g) {
                    const uint32_t b = __ballot_sync(0xffffffffu, (m >> g) & 1u);
                    if (lane == g) word = b;
                }
                if (lane < ngrp && (!partial || base + 32 * lane < rows))
                    tbits[(base >> 5) + lane] = partial ? word & tail_mask(base + 32 * lane, rows) : word;
            }
        }
    }
    __device__ __forceinline__ void store(Slots& r) {
#pragma unroll
        for (int k = 0; k < SCAN_STATE_SLOTS; ++k) r[k] = 0;
        r[0] = cnt;
    }
};

// ---- general predicate evaluator: per-lane numeric temporaries, warp-uniform NULL/TRUE/FALSE masks ----
constexpr int PG = PRED_GROUPS;

struct NumVal {
    uint64_t v[PG];    // per-lane payload, group g = tile row (base + 32 g + lane)
    uint32_t nul[PG];  // warp-uniform NULL masks
};
struct BoolVal {
    uint32_t t[PG], f[PG];  // warp-uniform TRUE / FALSE masks (neither bit set = NULL)
};

__device__ __forceinline__ void fetch_num(const ScanTables& P, const uint8_t* stage, uint8_t kind, uint16_t idx,
                                          uint64_t imm, const NumVal (&nt)[4], int row, NumVal& out) {
    if (kind == PK_NTEMP) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (k == idx) out = nt[k];
    } else if (kind == PK_IMM) {
#pragma unroll
        for (int g = 0; g < PG; ++g) {
            out.v[g] = imm;
            out.nul[g] = 0u;
        }
    } else if (kind == PK_NNULL) {
#pragma unroll
        for (int g = 0; g < PG; ++g) {
            out.v[g] = 0;
            out.nul[g] = 0xffffffffu;
        }
    } else {
        const ScanColDesc& c = P.cols[idx];
        const uint64_t* vals = reinterpret_cast<const uint64_t*>(stage + c.smem_val_off) + row;
#pragma unroll
        for (int g = 0; g < PG; ++g) {
            const uint64_t raw = vals[32 * g];
            out.v[g] = (kind == PK_COL_I64_AS_F64) ? d2u((double)(int64_t)raw) : raw;
            out.nul[g] = ~vword(c, stage, (row >> 5) + g);
        }
    }
}

__device__ __forceinline__ void fetch_bool(const ScanTables& P, const uint8_t* stage, uint8_t kind, uint16_t idx,
                                           uint64_t imm, const BoolVal (&bt)[4], int row, BoolVal& out) {
    if (kind == PK_BTEMP) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (k == idx) out = bt[k];
    } else if (kind == PK_BIMM) {
#pragma unroll
        for (int g = 0; g < PG; ++g) {
            out.t[g] = imm ? 0xffffffffu : 0u;
            out.f[g] = imm ? 0u : 0xffffffffu;
        }
    } else if (kind == PK_COL_BOOL) {
        const ScanColDesc& c = P.cols[idx];
        const uint32_t* vals = reinterpret_cast<const uint32_t*>(stage + c.smem_val_off);
#pragma unroll
        for (int g = 0; g < PG; ++g) {
            const uint32_t ok = vword(c, stage, (row >> 5) + g), b = vals[(row >> 5) + g];
            out.t[g] = b & ok;
            out.f[g] = ~b & ok;
        }
    } else {  // PK_BNULL / PK_NONE
#pragma unroll
        for (int g = 0; g < PG; ++g) out.t[g] = out.f[g] = 0u;
    }
}

// the two select-type instructions of numeric CASE / COALESCE, kept out of line: the evaluator's common instructions (and
// with them the register allocation of the scan kernel that calls it) stay exactly what they were without them
__device__ __noinline__ void pred_select(const ScanTables& P, const uint8_t* stage, const PredInstr& ins, NumVal (&nt)[4], const BoolVal (&bt)[4],
                                         int row, int lane) {
    NumVal a;
    fetch_num(P, stage, ins.a_kind, ins.a_idx, ins.imm, nt, row, a);
    if (ins.op == PO_KEEPIF_N) {
        BoolVal b;
        fetch_bool(P, stage, ins.b_kind, ins.b_idx, ins.imm, bt, row, b);
#pragma unroll
        for (int g = 0; g < PG; ++g) a.nul[g] |= ~b.t[g];
    } else {
        NumVal b;
        fetch_num(P, stage, ins.b_kind, ins.b_idx, ins.imm, nt, row, b);
#pragma unroll
        for (int g = 0; g < PG; ++g) {
            if ((a.nul[g] >> lane) & 1u) a.v[g] = b.v[g];
            a.nul[g] &= b.nul[g];
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (k == ins.dst) nt[k] = a;
}

// MASK: lane 0 also stores the TRUE word of every 32 rows to bits[] (bits[0] = the word of the unit's first row in this tile)
template <bool MASK>
__device__ __noinline__ void unit_pred(const ScanTables& P, const ScanUnitDesc& u, const uint8_t* stage, int lane,
                                       int rows_in_tile, uint64_t* cnt_out, uint64_t* div0_out, uint32_t* bits) {
    uint64_t cnt = 0;
    uint32_t div0 = 0;
    const int nw = u.nrows >> 5;
    for (int j = 0; j < nw; j += PG) {
        NumVal nt[4];
        BoolVal bt[4];
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int g = 0; g < PG; ++g) {
                nt[k].v[g] = 0;
                nt[k].nul[g] = 0xffffffffu;
                bt[k].t[g] = bt[k].f[g] = 0u;
            }
        const int row = u.row0 + 32 * j + lane;  // this lane's row in group 0
        for (int pc = 0; pc < u.code_len; ++pc) {
            const PredInstr ins = P.code[u.code_off + pc];
            if (ins.op < PO_ISNULL_N) {
                NumVal a, b;
                fetch_num(P, stage, ins.a_kind, ins.a_idx, ins.imm, nt, row, a);
                if (ins.b_kind != PK_NONE) fetch_num(P, stage, ins.b_kind, ins.b_idx, ins.imm, nt, row, b);
                else b = a;
                if (ins.op < PO_EQ_F) {
                    NumVal r;
#pragma unroll
                    for (int g = 0; g < PG; ++g) {
                        const double af = u2d(a.v[g]), bf = u2d(b.v[g]);
                        const int64_t ai = (int64_t)a.v[g], bi = (int64_t)b.v[g];
                        uint32_t nm = a.nul[g] | b.nul[g];
                        uint64_t o = 0;
                        switch (ins.op) {
                            case PO_MOVN: o = a.v[g]; break;
                            case PO_ADD_F: o = d2u(af + bf); break;
                            case PO_SUB_F: o = d2u(af - bf); break;
                            case PO_MUL_F: o = d2u(af * bf); break;
                            case PO_DIV_F: o = d2u(af / bf); break;
                            case PO_NEG_F: o = d2u(-af); break;
                            case PO_ABS_F: o = d2u(fabs(af)); break;
                            case PO_ADD_I: o = (uint64_t)ai + (uint64_t)bi; break;
                            case PO_SUB_I: o = (uint64_t)ai - (uint64_t)bi; break;
                            case PO_MUL_I: o = (uint64_t)ai * (uint64_t)bi; break;
                            case PO_DIV_I:
                            case PO_MOD_I: {
                                // (rows past the end of the table are zero padding: a column without a validity bitmap has
                                // no NULL bits to hide them, so they are masked here like in the final count)
                                const uint32_t z = __ballot_sync(0xffffffffu, bi == 0) & ~nm & tail_mask(u.row0 + 32 * (j + g), rows_in_tile);
                                div0 |= z;
                                nm |= z;
                                const int64_t sb = bi == 0 ? 1 : bi;
                                if (ins.op == PO_DIV_I) o = sb == -1 ? (uint64_t)0 - (uint64_t)ai : (uint64_t)(ai / sb);
                                else o = sb == -1 ? 0 : (uint64_t)(ai % sb);
                            } break;
                            case PO_NEG_I: o = (uint64_t)0 - (uint64_t)ai; break;
                            case PO_ABS_I: o = ai < 0 ? (uint64_t)0 - (uint64_t)ai : (uint64_t)ai; break;
                            case PO_I2F: o = d2u((double)ai); break;
                            default: break;
                        }
                        r.v[g] = o;
                        r.nul[g] = nm;
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (k == ins.dst) nt[k] = r;
                } else {
                    BoolVal r;
#pragma unroll
                    for (int g = 0; g < PG; ++g) {
                        const double af = u2d(a.v[g]), bf = u2d(b.v[g]);
                        const int64_t ai = (int64_t)a.v[g], bi = (int64_t)b.v[g];
                        bool c = false;
                        switch (ins.op) {
                            case PO_EQ_F: c = af == bf; break;
                            case PO_NE_F: c = af != bf; break;
                            case PO_LT_F: c = af < bf; break;
                            case PO_LE_F: c = af <= bf; break;
                            case PO_GT_F: c = af > bf; break;
                            case PO_GE_F: c = af >= bf; break;
                            case PO_EQ_I: c = ai == bi; break;
                            case PO_NE_I: c = ai != bi; break;
                            case PO_LT_I: c = ai < bi; break;
                            case PO_LE_I: c = ai <= bi; break;
                            case PO_GT_I: c = ai > bi; break;
                            case PO_GE_I: c = ai >= bi; break;
                            default: break;
                        }
                        const uint32_t m = __ballot_sync(0xffffffffu, c), known = ~(a.nul[g] | b.nul[g]);
                        r.t[g] = m & known;
                        r.f[g] = ~m & known;
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (k == ins.dst) bt[k] = r;
                }
            } else if (ins.op <= PO_ISNOTNULL_N) {
                NumVal a;
                fetch_num(P, stage, ins.a_kind, ins.a_idx, ins.imm, nt, row, a);
                BoolVal r;
#pragma unroll
                for (int g = 0; g < PG; ++g) {
                    r.t[g] = ins.op == PO_ISNULL_N ? a.nul[g] : ~a.nul[g];
                    r.f[g] = ~r.t[g];
                }
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (k == ins.dst) bt[k] = r;
            } else if (ins.op >= PO_KEEPIF_N) {
                pred_select(P, stage, ins, nt, bt, row, lane);
            } else {
                BoolVal a, b, r;
                fetch_bool(P, stage, ins.a_kind, ins.a_idx, ins.imm, bt, row, a);
                fetch_bool(P, stage, ins.b_kind, ins.b_idx, ins.imm, bt, row, b);
#pragma unroll
                for (int g = 0; g < PG; ++g) {
                    const uint32_t at = a.t[g], af = a.f[g], btt = b.t[g], bf = b.f[g];
                    uint32_t t = 0, f = 0;
                    switch (ins.op) {
                        case PO_MOVB: t = at; f = af; break;
                        case PO_AND: t = at & btt; f = af | bf; break;
                        case PO_OR: t = at | btt; f = af & bf; break;
                        case PO_NOT: t = af; f = at; break;
                        case PO_ISNULL_B: t = ~(at | af); f = at | af; break;
                        case PO_ISNOTNULL_B: t = at | af; f = ~(at | af); break;
                        case PO_ISTRUE: t = at; f = ~at; break;
                        case PO_ISFALSE: t = af; f = ~af; break;
                        case PO_EQ_B: t = (at & btt) | (af & bf); f = (at & bf) | (af & btt); break;
                        case PO_NE_B: t = (at & bf) | (af & btt); f = (at & btt) | (af & bf); break;
                        default: break;
                    }
                    r.t[g] = t;
                    r.f[g] = f;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (k == ins.dst) bt[k] = r;
            }
        }
#pragma unroll
        for (int g = 0; g < PG; ++g) {
            const uint32_t tw = bt[0].t[g] & tail_mask(u.row0 + 32 * (j + g), rows_in_tile);
            cnt += __popc(tw);
            if constexpr (MASK)
                if (bits && lane == 0 && u.row0 + 32 * (j + g) < rows_in_tile) bits[j + g] = tw;
        }
    }
    // masks are warp-uniform: lane 0 carries the counts
    if (lane == 0) {
        *cnt_out += cnt;
        *div0_out |= (uint64_t)(div0 != 0);
    }
}


template <bool MASK_>
struct PredUnit {
    static constexpr bool MASK = MASK_;
    const ScanTables* T;
    const ScanUnitDesc* u;
    int lane;
    uint64_t cnt, div0;
    uint32_t* tbits;
    __device__ __forceinline__ void at_tile(int64_t tile_row0) { tbits = u->bits ? u->bits + ((tile_row0 + u->row0) >> 5) : nullptr; }
    __device__ __forceinline__ void setup(const ScanTables& T_, const ScanUnitDesc& u_, int lane_) {
        T = &T_;
        u = &u_;
        lane = lane_;
    }
    __device__ __forceinline__ void load(const Slots& r) {
        cnt = r[0];
        div0 = r[1];
    }
    __device__ __forceinline__ void tile(const uint8_t* stage, int rows, bool) {
        unit_pred<MASK>(*T, *u, stage, lane, rows, &cnt, &div0, MASK ? tbits : nullptr);
    }
    __device__ __forceinline__ void store(Slots& r) {
#pragma unroll
        for (int k = 0; k < SCAN_STATE_SLOTS; ++k) r[k] = 0;
        r[0] = cnt;
        r[1] = div0;
    }
};

// reduce op of a state slot: 0 u64 add, 1 f64 add, 2 f64 min, 3 f64 max, 4 i64 min, 5 i64 max, 6 or
__host__ __device__ __forceinline__ int slot_op(int kind, int slot) {
    switch (kind) {
        case UNIT_COUNT: return 0;
        case UNIT_TERMS: return 0;
        case UNIT_PRED: return slot == 1 ? 6 : 0;
        case UNIT_PAIR: return slot == P_N ? 0 : 1;
        case UNIT_NUM_F64:
            if (slot == S_N || slot == S_ISUM) return 0;
            if (slot == S_MIN) return 2;
            if (slot == S_MAX) return 3;
            return 1;
        case UNIT_NUM_I64:
            if (slot == S_N || slot == S_ISUM) return 0;
            if (slot == S_MIN) return 4;
            if (slot == S_MAX) return 5;
            return 1;
    }
    return 0;
}
__device__ __forceinline__ uint64_t slot_combine(int op, uint64_t a, uint64_t b) {
    switch (op) {
        case 0: return a + b;
        case 1: return d2u(u2d(a) + u2d(b));
        case 2: return d2u(fmin(u2d(a), u2d(b)));
        case 3: return d2u(fmax(u2d(a), u2d(b)));
        case 4: return (uint64_t)min((int64_t)a, (int64_t)b);
        case 5: return (uint64_t)max((int64_t)a, (int64_t)b);
        default: return a | b;
    }
}
__host__ __device__ __forceinline__ uint64_t slot_identity(int kind, int slot) {
    int op = slot_op(kind, slot);
    switch (op) {
        case 2: return 0x7ff0000000000000ull;  // +inf
        case 3: return 0xfff0000000000000ull;  // -inf
        case 4: return (uint64_t)INT64_MAX;
        case 5: return (uint64_t)INT64_MIN;
        default: return 0;
    }
}

// cross-lane reduction of one unit's per-lane slots in a fixed butterfly order -> one record per (CTA, unit)
__device__ __forceinline__ void reduce_store(int kind, const Slots& r, uint64_t* out, int lane) {
#pragma unroll
    for (int sl = 0; sl < SCAN_STATE_SLOTS; ++sl) {
        const int op = slot_op(kind, sl);
        uint64_t v = r[sl];
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) v = slot_combine(op, v, shfl_xor_u64(v, m));
        if (lane == 0) out[sl] = v;
    }
}

// consumer-side view of the stage ring
struct Pipe {
    uint8_t* stages;
    uint64_t* full;
    uint64_t* empty;
    int n_stages, tile_rows;
    uint32_t stage_bytes;
    int64_t n_tiles;
    int64_t t_partial;  // index of the partial last tile, or -1
    int rows_partial;   // its row count
};

// a warp that owns exactly one unit: descriptors and accumulators live in registers for the whole scan
template <class U>
__device__ __forceinline__ void run_single(const Pipe& p, const ScanTables& T, const ScanUnitDesc& ud, uint64_t* out, int lane) {
    U unit;
    unit.setup(T, ud, lane);
    {
        Slots r;
#pragma unroll
        for (int k = 0; k < SCAN_STATE_SLOTS; ++k) r[k] = slot_identity(ud.kind, k);
        unit.load(r);
    }
    int s = 0;
    uint32_t ph = 0;
    for (int64_t t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
        mbar_wait(&p.full[s], ph);
        const bool partial = t == p.t_partial;
        if constexpr (U::MASK) unit.at_tile(t * p.tile_rows);
        unit.tile(p.stages + (size_t)s * p.stage_bytes, partial ? p.rows_partial : p.tile_rows, partial);
        __syncwarp();
        if (lane == 0) mbar_arrive(&p.empty[s]);
        if (++s == p.n_stages) {
            s = 0;
            ph ^= 1u;
        }
    }
    Slots r;
    unit.store(r);
    reduce_store(ud.kind, r, out, lane);
}
// a warp that owns several units: per-lane state lives in shared memory between tiles
template <class U>
__device__ __forceinline__ void run_once(const ScanTables& T, const ScanUnitDesc& ud, uint64_t* st, int lane, const uint8_t* stage,
                                         int rows, bool partial, int64_t tile_row0) {
    U unit;
    unit.setup(T, ud, lane);
    if constexpr (U::MASK) unit.at_tile(tile_row0);
    Slots r;
#pragma unroll
    for (int k = 0; k < SCAN_STATE_SLOTS; ++k) r[k] = st[k * 32 + lane];
    unit.load(r);
    unit.tile(stage, rows, partial);
    unit.store(r);
#pragma unroll
    for (int k = 0; k < SCAN_STATE_SLOTS; ++k) st[k * 32 + lane] = r[k];
}

// kind / flag dispatch, shared by both execution modes (SINGLE: whole tile loop inside; else one tile)
template <bool SINGLE, class U>
__device__ __forceinline__ void run_unit(const Pipe& p, const ScanTables& T, const ScanUnitDesc& ud, uint64_t* st, int lane,
                                         const uint8_t* stage, int rows, bool partial, int64_t tile_row0 = 0) {
    if (SINGLE) run_single<U>(p, T, ud, st, lane);
    else run_once<U>(T, ud, st, lane, stage, rows, partial, tile_row0);
}
template <bool SINGLE, bool IS_I64>
__device__ __forceinline__ void dispatch_num(const Pipe& p, const ScanTables& T, const ScanUnitDesc& ud, uint64_t* st, int lane,
                                             const uint8_t* stage, int rows, bool partial) {
    switch (ud.flags & 7) {
        case 0: run_unit<SINGLE, NumUnit<IS_I64, 0>>(p, T, ud, st, lane, stage, rows, partial); break;
        case 1: run_unit<SINGLE, NumUnit<IS_I64, 1>>(p, T, ud, st, lane, stage, rows, partial); break;
        case 2: run_unit<SINGLE, NumUnit<IS_I64, 2>>(p, T, ud, st, lane, stage, rows, partial); break;
        case 3: run_unit<SINGLE, NumUnit<IS_I64, 3>>(p, T, ud, st, lane, stage, rows, partial); break;
        case 4: run_unit<SINGLE, NumUnit<IS_I64, 4>>(p, T, ud, st, lane, stage, rows, partial); break;
        case 5: run_unit<SINGLE, NumUnit<IS_I64, 5>>(p, T, ud, st, lane, stage, rows, partial); break;
        case 6: run_unit<SINGLE, NumUnit<IS_I64, 6>>(p, T, ud, st, lane, stage, rows, partial); break;
        default: run_unit<SINGLE, NumUnit<IS_I64, 7>>(p, T, ud, st, lane, stage, rows, partial); break;
    }
}
// st: SINGLE -> global partial record of (CTA, unit); else this unit's per-lane state in shared memory
// MASKS: some unit of the pass writes row verdicts; its PRED / TERMS units store words where their descriptor has `bits`
template <bool SINGLE, bool MASKS>
__device__ __forceinline__ void dispatch_unit(const Pipe& p, const ScanTables& T, const ScanUnitDesc& ud, uint64_t* st, int lane,
                                              const uint8_t* stage, int rows, bool partial, int64_t tile_row0) {
    switch (ud.kind) {
        case UNIT_COUNT: run_unit<SINGLE, CountUnit>(p, T, ud, st, lane, stage, rows, partial); break;
        case UNIT_NUM_F64: dispatch_num<SINGLE, false>(p, T, ud, st, lane, stage, rows, partial); break;
        case UNIT_NUM_I64: dispatch_num<SINGLE, true>(p, T, ud, st, lane, stage, rows, partial); break;
        case UNIT_PAIR:
            switch ((ud.c0_is_i64 ? 1 : 0) | (ud.c1_is_i64 ? 2 : 0)) {
                case 0: run_unit<SINGLE, PairUnit<false, false>>(p, T, ud, st, lane, stage, rows, partial); break;
                case 1: run_unit<SINGLE, PairUnit<true, false>>(p, T, ud, st, lane, stage, rows, partial); break;
                case 2: run_unit<SINGLE, PairUnit<false, true>>(p, T, ud, st, lane, stage, rows, partial); break;
                default: run_unit<SINGLE, PairUnit<true, true>>(p, T, ud, st, lane, stage, rows, partial); break;
            }
            break;
        case UNIT_TERMS: run_unit<SINGLE, TermsUnit<MASKS>>(p, T, ud, st, lane, stage, rows, partial, tile_row0); break;
        default: run_unit<SINGLE, PredUnit<MASKS>>(p, T, ud, st, lane, stage, rows, partial, tile_row0); break;
    }
}

template <bool MASKS>
__global__ void __launch_bounds__(SCAN_THREADS, 1) scan_kernel(const __grid_constant__ ScanParams P) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* stages = scan_smem;
    uint64_t* state = reinterpret_cast<uint64_t*>(scan_smem + (size_t)P.n_stages * P.stage_bytes);
    uint64_t* full = state + (size_t)P.n_state_units * SCAN_STATE_SLOTS * 32;
    uint64_t* empty = full + P.n_stages;
    ScanTables* T = reinterpret_cast<ScanTables*>(empty + P.n_stages);

    // descriptor tables -> shared memory (only the used prefix of each array)
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&P.tab);
        uint32_t* dst = reinterpret_cast<uint32_t*>(T);
        auto copy = [&](size_t off, size_t bytes) {
            for (uint32_t i = threadIdx.x; i < bytes / 4; i += blockDim.x) dst[off / 4 + i] = src[off / 4 + i];
        };
        copy(offsetof(ScanTables, cols), sizeof(ScanColDesc) * P.n_cols);
        copy(offsetof(ScanTables, units), sizeof(ScanUnitDesc) * P.n_units);
        copy(offsetof(ScanTables, code), sizeof(PredInstr) * P.n_code);
        copy(offsetof(ScanTables, terms), sizeof(ScanTerm) * P.n_terms);
        copy(offsetof(ScanTables, warp_units), sizeof(T->warp_units));
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < P.n_stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], SCAN_CONSUMER_WARPS);
        }
        mbar_fence_init();
    }
    __syncthreads();
    const int rows_last = (int)(P.n_rows - (P.n_tiles - 1) * (int64_t)P.tile_rows);
    Pipe pipe{stages, full, empty, P.n_stages, P.tile_rows, P.stage_bytes, P.n_tiles,
              rows_last < P.tile_rows ? P.n_tiles - 1 : (int64_t)-1, rows_last};

    if (warp == 0) {
        // ---------------- TMA producer: lane c moves column c ----------------
        const bool active = lane < P.n_cols;
        const ScanColDesc c = T->cols[active ? lane : 0];
        const bool has_v = active && c.values != nullptr, has_b = active && c.validity != nullptr;
        int s = 0;
        uint32_t ph = 0;
        for (int64_t t = blockIdx.x; t < pipe.n_tiles; t += gridDim.x) {
            mbar_wait(&empty[s], ph ^ 1u);
            const int64_t row_base = t * pipe.tile_rows;
            const int rows = t == pipe.t_partial ? pipe.rows_partial : pipe.tile_rows;
            uint8_t* stage = stages + (size_t)s * pipe.stage_bytes;
            // byte counts padded to 16 (buffers are allocated with that slack)
            const uint32_t bbytes = has_b ? (uint32_t)(((rows + 7) / 8 + 15) & ~15) : 0u;
            const uint32_t vbytes = !has_v ? 0u : (c.kind == SC_BOOL ? (uint32_t)(((rows + 7) / 8 + 15) & ~15)
                                                                      : (uint32_t)((rows * 8 + 15) & ~15));
            uint32_t total = vbytes + bbytes;
#pragma unroll
            for (int m = 16; m > 0; m >>= 1) total += __shfl_xor_sync(0xffffffffu, total, m);
            if (lane == 0) mbar_arrive_expect_tx(&full[s], total);
            __syncwarp();
            if (vbytes) {
                const uint8_t* src = c.kind == SC_BOOL ? c.values + row_base / 8 : c.values + row_base * 8;
                bulk_g2s(stage + c.smem_val_off, src, vbytes, &full[s]);
            }
            if (bbytes) bulk_g2s(stage + c.smem_bits_off, c.validity + row_base / 8, bbytes, &full[s]);
            if (++s == pipe.n_stages) {
                s = 0;
                ph ^= 1u;
            }
        }
    } else {
        // ---------------- consumers ----------------
        const int cw = warp - 1;
        const int n_mine = T->warp_units[cw][0];
        if (P.n_state_units == 0) {
            // every warp owns at most one unit: registers only
            if (n_mine == 1) {
                const int u = T->warp_units[cw][1];
                dispatch_unit<true, MASKS>(pipe, *T, T->units[u], P.partials + ((size_t)blockIdx.x * P.n_units + u) * SCAN_STATE_SLOTS,
                                           lane, nullptr, 0, false, 0);
            } else {
                // idle warp: keep the ring moving
                int s = 0;
                uint32_t ph = 0;
                for (int64_t t = blockIdx.x; t < pipe.n_tiles; t += gridDim.x) {
                    mbar_wait(&full[s], ph);
                    if (lane == 0) mbar_arrive(&empty[s]);
                    if (++s == pipe.n_stages) {
                        s = 0;
                        ph ^= 1u;
                    }
                }
            }
        } else {
            for (int k = 0; k < n_mine; ++k) {
                const int u = T->warp_units[cw][1 + k];
                uint64_t* st = state + (size_t)u * SCAN_STATE_SLOTS * 32;
#pragma unroll
                for (int sl = 0; sl < SCAN_STATE_SLOTS; ++sl) st[sl * 32 + lane] = slot_identity(T->units[u].kind, sl);
            }
            __syncwarp();
            int s = 0;
            uint32_t ph = 0;
            for (int64_t t = blockIdx.x; t < pipe.n_tiles; t += gridDim.x) {
                mbar_wait(&full[s], ph);
                const bool partial = t == pipe.t_partial;
                const int rows = partial ? pipe.rows_partial : pipe.tile_rows;
                const uint8_t* stage = stages + (size_t)s * pipe.stage_bytes;
                for (int k = 0; k < n_mine; ++k) {
                    const int u = T->warp_units[cw][1 + k];
                    dispatch_unit<false, MASKS>(pipe, *T, T->units[u], state + (size_t)u * SCAN_STATE_SLOTS * 32, lane, stage, rows, partial,
                                                t * pipe.tile_rows);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[s]);
                if (++s == pipe.n_stages) {
                    s = 0;
                    ph ^= 1u;
                }
            }
            __syncwarp();
            for (int k = 0; k < n_mine; ++k) {
                const int u = T->warp_units[cw][1 + k];
                const uint64_t* st = state + (size_t)u * SCAN_STATE_SLOTS * 32;
                Slots r;
#pragma unroll
                for (int sl = 0; sl < SCAN_STATE_SLOTS; ++sl) r[sl] = st[sl * 32 + lane];
                reduce_store(T->units[u].kind, r, P.partials + ((size_t)blockIdx.x * P.n_units + u) * SCAN_STATE_SLOTS, lane);
            }
        }
    }
}

// one warp per aggregate: reduce partials[cta][unit] over CTAs and over the units feeding that aggregate
// One CTA per aggregate: thread i owns the (CTA b, unit u) partial records i, i+128, .. of that aggregate (all
// SCAN_STATE_SLOTS slots of a record are one 64-byte load, every load independent), then a fixed-shape
// shuffle + shared-memory tree combines them, so the result is bit-reproducible for a given (grid, plan).
constexpr int FIN_THREADS = 128;
__global__ void __launch_bounds__(FIN_THREADS) scan_finalize_kernel(const __grid_constant__ ScanParams P, int n_ctas, ScanAggOut* out) {
    const int agg = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __shared__ int ulist[SCAN_MAX_UNITS];
    __shared__ int s_nu, s_kind;
    __shared__ uint64_t red[FIN_THREADS / 32][SCAN_STATE_SLOTS];
    if (tid == 0) {
        int nu = 0, kind = -1;
        for (int u = 0; u < P.n_units; ++u)
            if (P.tab.units[u].agg == agg) {
                ulist[nu++] = u;
                kind = P.tab.units[u].kind;
            }
        s_nu = nu;
        s_kind = kind;
    }
    __syncthreads();
    const int nu = s_nu, kind = s_kind;
    if (kind < 0) return;
    uint64_t acc[SCAN_STATE_SLOTS];
    int op[SCAN_STATE_SLOTS];
#pragma unroll
    for (int k = 0; k < SCAN_STATE_SLOTS; ++k) {
        op[k] = slot_op(kind, k);
        acc[k] = slot_identity(kind, k);
    }
    const int total = n_ctas * nu;
    for (int i = tid; i < total; i += FIN_THREADS) {
        const int b = i / nu, u = ulist[i - b * nu];
        const ulonglong2* rec = reinterpret_cast<const ulonglong2*>(P.partials + ((size_t)b * P.n_units + u) * SCAN_STATE_SLOTS);
#pragma unroll
        for (int k = 0; k < SCAN_STATE_SLOTS / 2; ++k) {
            const ulonglong2 v = rec[k];
            acc[2 * k] = slot_combine(op[2 * k], acc[2 * k], v.x);
            acc[2 * k + 1] = slot_combine(op[2 * k + 1], acc[2 * k + 1], v.y);
        }
    }
#pragma unroll
    for (int k = 0; k < SCAN_STATE_SLOTS; ++k) {
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) acc[k] = slot_combine(op[k], acc[k], shfl_xor_u64(acc[k], m));
        if (lane == 0) red[warp][k] = acc[k];
    }
    __syncthreads();
    if (tid < SCAN_STATE_SLOTS) {
        uint64_t v = red[0][tid];
        const int o = slot_op(kind, tid);
        for (int w = 1; w < FIN_THREADS / 32; ++w) v = slot_combine(o, v, red[w][tid]);
        out[agg].s[tid] = v;
    }
}

// ---- host launchers (called from engine.cu) ----
size_t scan_smem_bytes(const ScanParams& P) {
    return (size_t)P.n_stages * P.stage_bytes + (size_t)P.n_state_units * SCAN_STATE_SLOTS * 32 * 8 +
           (size_t)2 * P.n_stages * 8 + sizeof(ScanTables);
}

cudaError_t scan_launch(const ScanParams& P, int grid, ScanAggOut* d_out, cudaStream_t stream) {
    size_t smem = scan_smem_bytes(P);
    // passes without requested row verdicts run the kernel that has no code for them
    bool masks = false;
    for (int u = 0; u < P.n_units; ++u) masks |= P.tab.units[u].bits != nullptr;
    const auto kernel = masks ? scan_kernel<true> : scan_kernel<false>;
    // the opt-in is per device (and per context): set it before every launch, it is a host-side table write
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    kernel<<<grid, SCAN_THREADS, smem, stream>>>(P);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    scan_finalize_kernel<<<P.n_aggs, FIN_THREADS, 0, stream>>>(P, grid, d_out);
    return cudaGetLastError();
}

}  // namespace tg
