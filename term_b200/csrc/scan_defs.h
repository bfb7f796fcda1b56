// Descriptors shared by the host planner and the fused numeric scan kernel (K1).
#pragma once
#include <stdint.h>

namespace tg {

constexpr int SCAN_MAX_COLS = 32;
constexpr int SCAN_MAX_UNITS = 48;
constexpr int SCAN_MAX_CODE = 128;
constexpr int SCAN_MAX_TERMS = 32;
constexpr int SCAN_UNIT_TERMS = 4;  // comparison terms a UNIT_TERMS unit keeps in registers
#ifndef TG_SCAN_CONSUMER_WARPS
#define TG_SCAN_CONSUMER_WARPS 16  // + 1 producer = 17 warps (96 registers per thread); measured against 15 @128 and 19 @96: best on both C2 suites
#endif
constexpr int SCAN_CONSUMER_WARPS = TG_SCAN_CONSUMER_WARPS;
constexpr int SCAN_THREADS = (SCAN_CONSUMER_WARPS + 1) * 32;  // warp 0 = TMA producer
constexpr int SCAN_STATE_SLOTS = 8;                           // 64-bit slots per lane per unit
constexpr int SCAN_MAX_STAGES = 8;
constexpr int SCAN_WARP_UNITS = 7;                            // units one consumer warp may own

// column kinds inside a tile
enum : int32_t { SC_F64 = 0, SC_I64 = 1, SC_BITS = 2 /* validity only */, SC_BOOL = 3 /* bit-packed values */ };

struct ScanColDesc {
    const uint8_t* values;    // device pointer or null (validity-only column)
    const uint8_t* validity;  // device pointer or null (no nulls)
    int32_t kind;
    uint32_t smem_val_off;   // byte offset of this column's values inside a stage
    uint32_t smem_bits_off;  // byte offset of its validity words inside a stage
    int32_t pivot_is_element;  // K is a valid value of the column: nulls may be replaced by K for min/max
    double pivot;            // shift K for the moment sums of this column
    int64_t ipivot;          // the same element as an integer (Int64 columns): pivot == (double)ipivot
};

enum : int32_t {
    UNIT_COUNT = 0,    // popcount of validity                -> slot0 = valid rows
    UNIT_NUM_F64 = 1,  // n, Σd, Σd², min, max   (Σx = n·K + Σd on the host)
    UNIT_NUM_I64 = 2,  // n, Σd, Σd², imin, imax, isum(wrapping); d = (double)x - K
    UNIT_PAIR = 3,     // n, Σdx, Σdy, Σdx², Σdy², Σdxdy over rows where both are valid
    UNIT_PRED = 4,     // slot0 = rows where predicate is TRUE, slot1 = integer division by zero seen
    UNIT_TERMS = 5,    // AND / OR of <= 4 `col cmp const` / IS [NOT] NULL terms: slot0 = TRUE rows
};

enum : int32_t { UF_MOMENTS = 1, UF_MINMAX = 2, UF_ISUM = 4 };

// slot meaning per unit kind (64-bit each)
enum : int32_t {
    S_N = 0,
    S_SD = 1,
    S_SDD = 2,
    S_MIN = 3,
    S_MAX = 4,
    S_SX = 5,
    S_ISUM = 6,
    // pair
    P_N = 0,
    P_SX = 1,
    P_SY = 2,
    P_SXX = 3,
    P_SYY = 4,
    P_SXY = 5,
};

struct ScanUnitDesc {
    int32_t kind;
    int32_t c0, c1;        // tile column indices
    int32_t row0, nrows;   // slice of the tile this unit covers (multiples of 64)
    int32_t agg;           // aggregate this unit accumulates into
    int32_t code_off, code_len;
    int32_t warp;          // owning consumer warp (0-based)
    int32_t c0_is_i64, c1_is_i64;  // pair units: convert on load
    int32_t flags;                 // NUM units: UF_MOMENTS | UF_MINMAX | UF_ISUM ; TERMS units: 1 = OR (else AND)
    uint32_t* bits;                // PRED / TERMS units of an aggregate whose row verdicts were requested: one TRUE word per
                                   // 32 rows of the table (word i = rows 32 i .. 32 i + 31), else null
};

// Predicate code (SQL three-valued logic) for the warp-mask evaluator:
//   numeric temporaries N0..N3 : one 64-bit payload per lane (row) + a warp-uniform 32-bit NULL mask
//   boolean temporaries B0..B3 : warp-uniform (TRUE mask, FALSE mask) pairs, bit l = row of lane l
// Comparisons are one per-lane compare + one ballot; AND/OR/NOT/IS NULL are 1-2 mask instructions
// for 32 rows at once. The predicate's value must end in B0.
constexpr int PRED_GROUPS = 2;  // 32-row groups evaluated per instruction decode
enum : uint8_t {
    PK_NTEMP = 0,
    PK_COL_F64 = 1,
    PK_COL_I64 = 2,
    PK_COL_I64_AS_F64 = 3,
    PK_IMM = 4,       // numeric immediate: imm bits (f64 or i64)
    PK_NNULL = 5,     // numeric NULL literal
    PK_BTEMP = 6,
    PK_COL_BOOL = 7,
    PK_BIMM = 8,      // boolean literal (imm 0/1)
    PK_BNULL = 9,     // boolean NULL
    PK_NONE = 10,
};
enum : uint8_t {
    // numeric -> numeric
    PO_MOVN = 0,
    PO_ADD_F, PO_SUB_F, PO_MUL_F, PO_DIV_F, PO_NEG_F, PO_ABS_F,
    PO_ADD_I, PO_SUB_I, PO_MUL_I, PO_DIV_I, PO_MOD_I, PO_NEG_I, PO_ABS_I,
    PO_I2F,
    // numeric -> boolean
    PO_EQ_F, PO_NE_F, PO_LT_F, PO_LE_F, PO_GT_F, PO_GE_F,
    PO_EQ_I, PO_NE_I, PO_LT_I, PO_LE_I, PO_GT_I, PO_GE_I,
    PO_ISNULL_N, PO_ISNOTNULL_N,
    // boolean -> boolean
    PO_MOVB, PO_AND, PO_OR, PO_NOT, PO_ISNULL_B, PO_ISNOTNULL_B, PO_ISTRUE, PO_ISFALSE, PO_EQ_B, PO_NE_B,
    // (numeric a, boolean b) -> numeric: a where b is TRUE, NULL elsewhere (the arms of a numeric CASE)
    PO_KEEPIF_N,
    // (numeric a, numeric b) -> numeric: a unless it is NULL, else b (same numeric type on both sides)
    PO_COALESCE_N,
};
struct PredInstr {
    uint8_t op;
    uint8_t dst;     // temp index 0..3 (numeric or boolean file, by op class)
    uint8_t a_kind, b_kind;
    uint16_t a_idx, b_idx;  // temp index or tile column index
    uint64_t imm;           // shared immediate (at most one of a/b is PK_IMM / PK_BIMM)
};
static_assert(sizeof(PredInstr) == 16, "PredInstr layout");

// One comparison term of a UNIT_TERMS unit: TRUE iff the row is valid and (x < c, x == c, x > c) selects
// a set bit of cmp_mask (bit0 lt, bit1 eq, bit2 gt); TK_ISNULL / TK_NOTNULL test validity only.
enum : int32_t { TK_F64 = 0, TK_I64 = 1, TK_I64_AS_F64 = 2, TK_ISNULL = 3, TK_NOTNULL = 4 };
struct ScanTerm {
    int32_t col;
    int32_t kind;
    int32_t cmp_mask;
    int32_t pad;
    uint64_t imm;
};

// descriptor tables: copied to shared memory at kernel start (uniform, low-latency access)
struct ScanTables {
    ScanColDesc cols[SCAN_MAX_COLS];
    ScanUnitDesc units[SCAN_MAX_UNITS];
    PredInstr code[SCAN_MAX_CODE];
    ScanTerm terms[SCAN_MAX_TERMS];
    int32_t warp_units[SCAN_CONSUMER_WARPS][SCAN_WARP_UNITS + 1];  // [w][0] = count, then unit ids
};

struct ScanParams {
    int64_t n_rows;
    int64_t n_tiles;
    int32_t tile_rows;
    int32_t n_cols;
    int32_t n_units;
    int32_t n_stages;
    uint32_t stage_bytes;
    int32_t n_aggs;
    int32_t n_code;
    int32_t n_terms;
    int32_t n_state_units;  // 0: every consumer warp owns <= 1 unit (state in registers); else n_units
    uint64_t* partials;  // [gridDim.x][n_units][SCAN_STATE_SLOTS]
    ScanTables tab;
};

// Result of the finalize kernel: one record per aggregate.
struct ScanAggOut {
    uint64_t s[SCAN_STATE_SLOTS];
};

}  // namespace tg
