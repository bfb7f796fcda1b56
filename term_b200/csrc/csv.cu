// CSV -> HBM: tokenize and parse whole records on the device into the Arrow layout. Replaces the CPU parse of the
// reference's CsvSource (sources/, registered through DataFusion's CSV reader, i.e. arrow-csv) and the host->device copy.
//
// The host stages the file through the pinned ring in chunks of TG_CSV_CHUNK_BYTES (default 256 MiB), double-buffered:
// window k + 1 is uploaded on a side stream while the kernels of chunk k run on the copy stream. Every chunk starts at a
// record boundary; the part of a record a chunk cuts off is copied (device to device) in front of the next window.
//   K8a tokenizer   the quoting state machine (field start / unquoted / quoted / quote seen in quoted) run as a scan of
//                   transition vectors: pass 1 composes every tile's 4-entry map and its separator counts per start state,
//                   one CTA scans the tiles, pass 2 re-runs each thread from its true state and writes the positions of
//                   the unquoted delimiters and record terminators (a terminator right after a terminator byte — blank
//                   lines, the LF of a CRLF — is not one). Record r of K columns owns separators [rK, rK + K), so the
//                   field count check is one test per separator.
//   K8b parsers     one kernel per stored type, one warp per 32 records: the value into the column's reserved tail, a
//                   chunk-relative validity word per ballot, NULL counts by popcount, the first error by atomicMin on the
//                   field index. Float64 is exact (Clinger's fast path, then Eisel-Lemire over a 128-bit power-of-five
//                   table); a field it cannot decide goes to a fallback list the host re-parses with strtod. Utf8 fields
//                   are unescaped in place and validated, and the Parquet BYTE_ARRAY tail writes offsets and bytes.
// Any other dialect (quote, escape, comment or terminator bytes, a NULL regex) runs the general 7-state machine from a
// byte-indexed transition table built on the host, and parsers that unescape every field and test the NULL regex's DFA.
// One read-back per chunk (records, bytes consumed, first error, NULL counts, fallback count, the pivot's head values);
// Utf8 columns add the byte total read inside append_utf8_from_entries.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "engine.hpp"
#include "regex_dfa.hpp"
#include "str_entries.cuh"

namespace tg {

#define HD __host__ __device__ __forceinline__

// ---------------------------------------------------------------------------------------------------------------------
// value parsers (host and device: tg_csv_parse_value runs the same code on the CPU)
// ---------------------------------------------------------------------------------------------------------------------
enum CsvKind : int32_t { CSV_I64, CSV_I32, CSV_F64, CSV_BOOL, CSV_UTF8, CSV_DATE32, CSV_TS };
enum CsvStatus : int32_t { CSV_OK = 0, CSV_NULL, CSV_BAD, CSV_RANGE, CSV_SLOW /* Float64: needs the exact slow path */, CSV_BADUTF8, CSV_LONG };

// a field's text after unquoting: `a` then `b` (a quoted field: the part inside the quotes, then the bytes after the
// closing quote, kept literally). A value of a non-string type cannot hold a quote, so `""` inside one is an error.
struct CsvText {
    const uint8_t* a;
    uint32_t na;
    const uint8_t* b;
    uint32_t nb;
    HD uint32_t size() const { return na + nb; }
    HD uint8_t operator[](uint32_t i) const { return i < na ? a[i] : b[i - na]; }
};

// false: the field holds a doubled quote (or no closing quote)
HD bool csv_text(const uint8_t* p, uint32_t n, CsvText& t) {
    t = CsvText{p, n, p, 0};
    if (n == 0 || p[0] != '"') return true;
    for (uint32_t i = 1; i < n; ++i)
        if (p[i] == '"') {
            if (i + 1 < n && p[i + 1] == '"') return false;
            t = CsvText{p + 1, i - 1, p + i + 1, n - i - 1};
            for (uint32_t k = 0; k < t.nb; ++k)
                if (t.b[k] == '"') return false;
            return true;
        }
    return false;
}

HD bool csv_ieq(const CsvText& t, uint32_t from, const char* lit) {
    uint32_t i = 0;
    for (; lit[i]; ++i) {
        if (from + i >= t.size()) return false;
        uint8_t c = t[from + i];
        if (c >= 'A' && c <= 'Z') c = (uint8_t)(c + 32);
        if (c != (uint8_t)lit[i]) return false;
    }
    return from + i == t.size();
}

HD int32_t csv_parse_int(const CsvText& t, bool is32, int64_t* out) {
    const uint32_t n = t.size();
    uint32_t i = 0;
    bool neg = false;
    if (n && (t[0] == '+' || t[0] == '-')) neg = t[i++] == '-';
    if (i == n) return CSV_BAD;
    uint64_t m = 0;
    bool over = false;
    for (; i < n; ++i) {
        const uint32_t d = (uint32_t)t[i] - '0';
        if (d > 9) return CSV_BAD;
        if (m > (~0ull - d) / 10) over = true;
        else m = m * 10 + d;
    }
    const uint64_t lim = is32 ? (neg ? 2147483648ull : 2147483647ull) : (neg ? 9223372036854775808ull : 9223372036854775807ull);
    if (over || m > lim) return CSV_RANGE;
    *out = neg ? (int64_t)(0ull - m) : (int64_t)m;
    return CSV_OK;
}

// ---- Float64 ----
#ifdef __CUDA_ARCH__
#define CSV_POW5 CSV_POW5_D
#else
#define CSV_POW5 CSV_POW5_H
#endif
__device__ const uint64_t CSV_POW5_D[][2] = {
#include "pow5_128.inc"
};
#ifndef __CUDA_ARCH__
static const uint64_t CSV_POW5_H[][2] = {
#include "pow5_128.inc"
};
#endif
constexpr int CSV_Q_MIN = -342, CSV_Q_MAX = 308;

HD void csv_mul128(uint64_t a, uint64_t b, uint64_t* hi, uint64_t* lo) {
#ifdef __CUDA_ARCH__
    *hi = __umul64hi(a, b);
    *lo = a * b;
#else
    const unsigned __int128 p = (unsigned __int128)a * b;
    *hi = (uint64_t)(p >> 64);
    *lo = (uint64_t)p;
#endif
}

HD int csv_clz(uint64_t w) {
#ifdef __CUDA_ARCH__
    return __clzll((long long)w);
#else
    return __builtin_clzll(w);
#endif
}

HD uint64_t csv_pow5(int q, int half) {
#ifdef __CUDA_ARCH__
    return __ldg(&CSV_POW5[q - CSV_Q_MIN][half]);
#else
    return CSV_POW5[q - CSV_Q_MIN][half];
#endif
}

// w * 10^q (w != 0) correctly rounded, as IEEE bits without the sign: Eisel-Lemire with the 128-bit product, which decides
// every 64-bit w (Mushtak & Lemire 2023); the structure follows fast_float's compute_float<binary64>
HD uint64_t csv_eisel_lemire(uint64_t w, int64_t q) {
    if (q < CSV_Q_MIN) return 0;
    if (q > CSV_Q_MAX) return 0x7FFull << 52;
    const int lz = csv_clz(w);
    w <<= lz;
    uint64_t hi, lo;
    csv_mul128(w, csv_pow5((int)q, 0), &hi, &lo);
    const uint64_t mask = 0xFFFFFFFFFFFFFFFFull >> 55;  // 52 + 3 bits of precision
    if ((hi & mask) == mask) {
        uint64_t hi2, lo2;
        csv_mul128(w, csv_pow5((int)q, 1), &hi2, &lo2);
        lo += hi2;
        if (hi2 > lo) ++hi;
    }
    const int upper = (int)(hi >> 63);
    const int shift = upper + 64 - 52 - 3;
    uint64_t mant = hi >> shift;
    int32_t p2 = (int32_t)(((((152170 + 65536) * (int32_t)q) >> 16) + 63) + upper - lz + 1023);
    if (p2 <= 0) {  // subnormal
        if (-p2 + 1 >= 64) return 0;
        mant >>= -p2 + 1;
        mant += mant & 1;
        mant >>= 1;
        p2 = mant < (1ull << 52) ? 0 : 1;
        return (mant & ~(1ull << 52)) | ((uint64_t)p2 << 52);
    }
    // exactly between two floats (only possible while 5^q fits 64 bits): round to even
    if (lo <= 1 && q >= -4 && q <= 23 && (mant & 3) == 1 && (mant << shift) == hi) mant &= ~1ull;
    mant += mant & 1;
    mant >>= 1;
    if (mant >= (2ull << 52)) {
        mant = 1ull << 52;
        ++p2;
    }
    mant &= ~(1ull << 52);
    if (p2 >= 0x7FF) return 0x7FFull << 52;
    return mant | ((uint64_t)p2 << 52);
}

HD uint64_t csv_decimal_bits(uint64_t w, int64_t q) {
    // Clinger: w and 10^|q| are exact doubles, so one correctly rounded product / quotient is the answer
    if (w <= (1ull << 53) && q >= -22 && q <= 22) {
        double p = 1.0;
        for (int i = 0; i < (q < 0 ? -q : q); ++i) p *= 10.0;  // exact: 10^22 < 2^53 * 2^22
#ifdef __CUDA_ARCH__
        const double d = q < 0 ? __ddiv_rn((double)w, p) : __dmul_rn((double)w, p);
        return (uint64_t)__double_as_longlong(d);
#else
        const double d = q < 0 ? (double)w / p : (double)w * p;
        uint64_t b;
        memcpy(&b, &d, 8);
        return b;
#endif
    }
    return csv_eisel_lemire(w, q);
}

// grammar [+-]?(digits[.digits?] | .digits)([eE][+-]?digits)? and [+-]?(nan | inf | infinity), case-insensitive;
// CSV_SLOW: more than 19 significant digits and the first 19 (w) and w + 1 round differently
HD int32_t csv_parse_f64(const CsvText& t, uint64_t* bits) {
    const uint32_t n = t.size();
    uint32_t i = 0;
    bool neg = false;
    if (n && (t[0] == '+' || t[0] == '-')) neg = t[i++] == '-';
    const uint64_t sign = neg ? 1ull << 63 : 0;
    if (csv_ieq(t, i, "nan")) {
        *bits = sign | 0x7FF8000000000000ull;
        return CSV_OK;
    }
    if (csv_ieq(t, i, "inf") || csv_ieq(t, i, "infinity")) {
        *bits = sign | (0x7FFull << 52);
        return CSV_OK;
    }
    uint64_t w = 0;
    int nd = 0, digits = 0;
    int64_t q = 0;
    bool dropped = false;
    for (; i < n && (uint32_t)t[i] - '0' <= 9; ++i, ++digits) {
        const uint32_t d = (uint32_t)t[i] - '0';
        if (w == 0 && d == 0) continue;
        if (nd < 19) w = w * 10 + d, ++nd;
        else ++q, dropped |= d != 0;
    }
    if (i < n && t[i] == '.') {
        for (++i; i < n && (uint32_t)t[i] - '0' <= 9; ++i, ++digits) {
            const uint32_t d = (uint32_t)t[i] - '0';
            if (w == 0 && d == 0) --q;
            else if (nd < 19) w = w * 10 + d, ++nd, --q;
            else dropped |= d != 0;
        }
    }
    if (digits == 0) return CSV_BAD;
    if (i < n && (t[i] == 'e' || t[i] == 'E')) {
        ++i;
        bool eneg = false;
        if (i < n && (t[i] == '+' || t[i] == '-')) eneg = t[i++] == '-';
        int64_t ex = 0;
        int ed = 0;
        for (; i < n && (uint32_t)t[i] - '0' <= 9; ++i, ++ed)
            if (ex < 100000000) ex = ex * 10 + (t[i] - '0');
        if (ed == 0) return CSV_BAD;
        q += eneg ? -ex : ex;
    }
    if (i != n) return CSV_BAD;
    if (w == 0) {
        *bits = sign;
        return CSV_OK;
    }
    const uint64_t b = csv_decimal_bits(w, q);
    if (dropped && csv_decimal_bits(w + 1, q) != b) return CSV_SLOW;
    *bits = sign | b;
    return CSV_OK;
}

// ---- Boolean / Date32 / Timestamp ----
HD int32_t csv_parse_bool(const CsvText& t, uint32_t* v) {
    if (csv_ieq(t, 0, "true")) return *v = 1, CSV_OK;
    if (csv_ieq(t, 0, "false")) return *v = 0, CSV_OK;
    return CSV_BAD;
}

HD bool csv_digits(const CsvText& t, uint32_t at, int n, int32_t* v) {
    int32_t x = 0;
    for (int k = 0; k < n; ++k) {
        const uint32_t d = (uint32_t)t[at + k] - '0';
        if (d > 9) return false;
        x = x * 10 + (int32_t)d;
    }
    *v = x;
    return true;
}

// days since 1970-01-01 of a proleptic Gregorian date (H. Hinnant's days_from_civil)
HD int64_t csv_days_from_civil(int64_t y, int64_t m, int64_t d) {
    y -= m <= 2;
    const int64_t era = (y >= 0 ? y : y - 399) / 400;
    const int64_t yoe = y - era * 400;
    const int64_t doy = (153 * (m + (m > 2 ? -3 : 9)) + 2) / 5 + d - 1;
    const int64_t doe = yoe * 365 + yoe / 4 - yoe / 100 + doy;
    return era * 146097 + doe - 719468;
}

// YYYY-MM-DD at t[0..10)
HD bool csv_date(const CsvText& t, int64_t* days) {
    int32_t y, m, d;
    if (t.size() < 10 || t[4] != '-' || t[7] != '-' || !csv_digits(t, 0, 4, &y) || !csv_digits(t, 5, 2, &m) || !csv_digits(t, 8, 2, &d)) return false;
    if (m < 1 || m > 12 || d < 1) return false;
    const bool leap = (y % 4 == 0 && y % 100 != 0) || y % 400 == 0;
    const int dim = m == 2 ? (leap ? 29 : 28) : (m == 4 || m == 6 || m == 9 || m == 11) ? 30 : 31;
    if (d > dim) return false;
    *days = csv_days_from_civil(y, m, d);
    return true;
}

HD int32_t csv_parse_date32(const CsvText& t, int64_t* out) {
    return t.size() == 10 && csv_date(t, out) ? CSV_OK : CSV_BAD;
}

// YYYY-MM-DD[T| ]HH:MM:SS[.f{1,9}], naive; unit 's' / 'm' / 'u' / 'n'; fraction digits past the unit are dropped (floor)
HD int32_t csv_parse_ts(const CsvText& t, char unit, int64_t* out) {
    const uint32_t n = t.size();
    int64_t days;
    int32_t hh, mm, ss;
    if (n < 19 || !csv_date(t, &days) || (t[10] != 'T' && t[10] != ' ') || t[13] != ':' || t[16] != ':' || !csv_digits(t, 11, 2, &hh) ||
        !csv_digits(t, 14, 2, &mm) || !csv_digits(t, 17, 2, &ss) || hh > 23 || mm > 59 || ss > 59)
        return CSV_BAD;
    // the fraction in the unit: its first 0 / 3 / 6 / 9 digits, padded with zeros
    const int ud = unit == 's' ? 0 : unit == 'm' ? 3 : unit == 'u' ? 6 : 9;
    int64_t frac = 0;
    int fd = 0;
    if (n > 19) {
        if (t[19] != '.' || n < 21 || n > 29) return CSV_BAD;
        for (uint32_t i = 20; i < n; ++i) {
            const uint32_t d = (uint32_t)t[i] - '0';
            if (d > 9) return CSV_BAD;
            if (fd < ud) frac = frac * 10 + d, ++fd;
        }
    }
    for (; fd < ud; ++fd) frac *= 10;
    const int64_t per_s = unit == 's' ? 1 : unit == 'm' ? 1000 : unit == 'u' ? 1000000 : 1000000000;
    const __int128 v = ((__int128)days * 86400 + hh * 3600 + mm * 60 + ss) * per_s + frac;
    if (v > (__int128)9223372036854775807ll || v < -(__int128)9223372036854775807ll - 1) return CSV_RANGE;
    *out = (int64_t)v;
    return CSV_OK;
}

// ---- Utf8 ----
// valid UTF-8 (no overlong forms, surrogates or code points above U+10FFFF)
HD bool csv_utf8_valid(const uint8_t* p, uint32_t n) {
    uint32_t i = 0;
    while (i < n) {
        const uint8_t c = p[i];
        if (c < 0x80) {
            ++i;
            continue;
        }
        int more;
        uint8_t lo = 0x80, hi = 0xBF;
        if (c >= 0xC2 && c <= 0xDF) more = 1;
        else if (c == 0xE0) more = 2, lo = 0xA0;
        else if (c == 0xED) more = 2, hi = 0x9F;
        else if (c >= 0xE1 && c <= 0xEF) more = 2;
        else if (c == 0xF0) more = 3, lo = 0x90;
        else if (c == 0xF4) more = 3, hi = 0x8F;
        else if (c >= 0xF1 && c <= 0xF3) more = 3;
        else return false;
        if (i + (uint32_t)more >= n) return false;
        if (p[i + 1] < lo || p[i + 1] > hi) return false;
        for (int k = 2; k <= more; ++k)
            if (p[i + k] < 0x80 || p[i + k] > 0xBF) return false;
        i += (uint32_t)more + 1;
    }
    return true;
}

// unescapes a field in place (`dst` may equal `p`: the result is never longer) and returns its length. Inside quotes a
// doubled quote is one quote and the escape byte (esc >= 0) stands for the byte after it; bytes after the closing quote
// and an unquoted field are kept as they are.
HD uint32_t csv_unescape(const uint8_t* p, uint32_t n, uint8_t* dst, int32_t quote = '"', int32_t esc = -1) {
    if (n == 0 || p[0] != quote) {
        if (dst != p)
            for (uint32_t i = 0; i < n; ++i) dst[i] = p[i];
        return n;
    }
    uint32_t o = 0;
    int st = 2;  // 2 quoted, 3 quote seen, 1 after the closing quote, 4 escape seen
    for (uint32_t i = 1; i < n; ++i) {
        const uint8_t c = p[i];
        if (st == 2) {
            if (c == quote) st = 3;
            else if (c == esc) st = 4;
            else dst[o++] = c;
        } else if (st == 4) {
            dst[o++] = c;
            st = 2;
        } else if (st == 3) {
            dst[o++] = c;
            st = c == quote ? 2 : 1;
        } else {
            dst[o++] = c;
        }
    }
    return o;
}

// a non-string value's text -> its stored value (8 bytes; Int32 / Date32 in the low 4, Boolean 0 / 1)
HD int32_t csv_parse_text(int32_t kind, char unit, const CsvText& t, uint64_t* v) {
    int64_t x = 0;
    int32_t st;
    switch (kind) {
        case CSV_I64: st = csv_parse_int(t, false, &x); break;
        case CSV_I32: st = csv_parse_int(t, true, &x); break;
        case CSV_F64: return csv_parse_f64(t, v);
        case CSV_BOOL: {
            uint32_t b = 0;
            st = csv_parse_bool(t, &b);
            x = b;
        } break;
        case CSV_DATE32: st = csv_parse_date32(t, &x); break;
        default: st = csv_parse_ts(t, unit, &x); break;
    }
    *v = (uint64_t)x;
    return st;
}

// one raw non-string field of the default format: an empty field, quoted or not, is NULL
HD int32_t csv_parse_fixed(int32_t kind, char unit, const uint8_t* p, uint32_t n, uint64_t* v) {
    CsvText t;
    if (!csv_text(p, n, t)) return CSV_BAD;
    if (t.size() == 0) return CSV_NULL;
    return csv_parse_text(kind, unit, t, v);
}

// ---- formats with other quote, escape, comment or terminator bytes, or a NULL regex
struct CsvFieldFmt {
    int32_t quote, esc, comment, term;  // esc / comment: -1 none; term: -1 LF, CRLF or a lone CR
    const uint8_t* null_tab;            // the NULL regex (csv_null_table), or nullptr: an empty field is NULL
};

HD bool csv_is_term(uint8_t c, int32_t term) { return term < 0 ? (c == '\n' || c == '\r') : c == term; }

// the first byte of a record's first field in [a, e): blank records and comment lines before it are skipped
HD uint32_t csv_record_start(const uint8_t* p, uint32_t a, uint32_t e, int32_t comment, int32_t term) {
    while (a < e) {
        if (csv_is_term(p[a], term)) ++a;
        else if (p[a] == comment)
            while (a < e && !csv_is_term(p[a], term)) ++a;
        else break;
    }
    return a;
}

// the NULL regex's DFA (regex_dfa.cpp) as one table: n_classes, start state (uint32 each, then 8 bytes of padding), the
// 256-entry byte class map, then one row per state of n_classes next states and an END entry (1: a haystack ending in
// this state matches), uint16 each, as strings.cu lays out its rows. Unanchored search, as Regex::is_match.
HD bool csv_null_match(const uint8_t* tab, const uint8_t* p, uint32_t n) {
    const uint32_t nc = reinterpret_cast<const uint32_t*>(tab)[0];
    uint32_t st = reinterpret_cast<const uint32_t*>(tab)[1];
    const uint8_t* cls = tab + 16;
    const uint16_t* rows = reinterpret_cast<const uint16_t*>(tab + 16 + 256);
    for (uint32_t i = 0; i < n && st > 1; ++i) st = rows[st * (nc + 1) + cls[p[i]]];
    return st == 1 || (st != 0 && rows[st * (nc + 1) + nc] != 0);  // 1 = DFA_MATCH, 0 = DFA_DEAD
}

// one raw field of a general format, unescaped in place: NULL when the regex finds a match in the unescaped value (no
// regex: when it is empty); otherwise the value (a non-NULL empty field is "" for Utf8 and a value error for the others)
HD int32_t csv_parse_general(int32_t kind, char unit, uint8_t* p, uint32_t n, const CsvFieldFmt& f, uint64_t* v, uint32_t* len) {
    const uint32_t m = csv_unescape(p, n, p, f.quote, f.esc);
    *len = m;
    if (f.null_tab ? csv_null_match(f.null_tab, p, m) : m == 0) return CSV_NULL;
    if (kind == CSV_UTF8) return m > PQ_STR_MAX_LEN ? CSV_LONG : csv_utf8_valid(p, m) ? CSV_OK : CSV_BADUTF8;
    return csv_parse_text(kind, unit, CsvText{p, m, p, 0}, v);
}

// ---------------------------------------------------------------------------------------------------------------------
// K8a tokenizer
// ---------------------------------------------------------------------------------------------------------------------
constexpr int CSV_THREADS = 256, CSV_BPT = 16, CSV_TILE = CSV_THREADS * CSV_BPT;
enum : uint32_t { ST_FIELD = 0, ST_UNQ = 1, ST_QUO = 2, ST_QSEEN = 3 };
// next state by byte class (other, quote, delimiter, terminator): one byte per class, 2 bits per current state
constexpr uint32_t CSV_NEXT = (ST_UNQ | ST_UNQ << 2 | ST_QUO << 4 | ST_UNQ << 6) |               // other
                              (ST_QUO | ST_UNQ << 2 | ST_QSEEN << 4 | ST_QUO << 6) << 8 |       // quote
                              (ST_FIELD | ST_FIELD << 2 | ST_QUO << 4 | ST_FIELD << 6) << 16 |  // delimiter
                              (ST_FIELD | ST_FIELD << 2 | ST_QUO << 4 | ST_FIELD << 6) << 24;   // terminator
__device__ __forceinline__ uint32_t csv_next(uint32_t cls) { return (CSV_NEXT >> (8 * cls)) & 0xFFu; }

// The general machine (any other format): 7 states, 3 bits each in a map. Every byte value has one transition word,
// built on the host from the format (csv_machine): bits [3s, 3s + 3) the next state from state s, bit 21 + s set when the
// byte ends a field from state s, bit 28 set when the byte is a record terminator. csv-core's reader: the comment byte
// counts only at a record's start, the escape byte only inside quotes; a terminator at a record's start is a blank record.
enum : uint32_t { G_REC = 0, G_FIELD = 1, G_UNQ = 2, G_QUO = 3, G_QSEEN = 4, G_ESC = 5, G_CMT = 6 };
constexpr int G_EMIT = 21, G_TERM = 28;

// bits per map entry and the number of start states of the 4-state (default format) and the general machine
__host__ __device__ constexpr int csv_sb(int ns) { return ns == 4 ? 2 : 3; }
template <int NS>
__host__ __device__ constexpr uint32_t csv_identity() {
    uint32_t m = 0;
    for (int s = 0; s < NS; ++s) m |= (uint32_t)s << (csv_sb(NS) * s);
    return m;
}
template <int NS>
__device__ __forceinline__ uint32_t csv_at(uint32_t map, uint32_t s) {
    return (map >> (csv_sb(NS) * s)) & ((1u << csv_sb(NS)) - 1);
}

// what a run of bytes does from each of the NS start states: the end state and the separators emitted
template <int NS>
struct CsvSeg {
    uint32_t map;
    uint32_t c[NS];
};
template <int NS>
__device__ __forceinline__ CsvSeg<NS> csv_seg_identity() {
    CsvSeg<NS> g;
    g.map = csv_identity<NS>();
#pragma unroll
    for (int s = 0; s < NS; ++s) g.c[s] = 0;
    return g;
}
template <int NS>
__device__ __forceinline__ CsvSeg<NS> csv_combine(const CsvSeg<NS>& a, const CsvSeg<NS>& b) {  // a, then b
    CsvSeg<NS> r;
    r.map = 0;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const uint32_t m = csv_at<NS>(a.map, s);
        r.map |= csv_at<NS>(b.map, m) << (csv_sb(NS) * s);
        r.c[s] = a.c[s] + b.c[m];
    }
    return r;
}
template <int NS>
__device__ __forceinline__ CsvSeg<NS> csv_shfl_up(const CsvSeg<NS>& x, int o) {
    CsvSeg<NS> r;
    r.map = __shfl_up_sync(0xffffffffu, x.map, o);
#pragma unroll
    for (int s = 0; s < NS; ++s) r.c[s] = __shfl_up_sync(0xffffffffu, x.c[s], o);
    return r;
}

__device__ __forceinline__ uint32_t csv_class(uint8_t c, uint8_t delim) {
    return c == '"' ? 1u : c == delim ? 2u : (c == '\n' || c == '\r') ? 3u : 0u;
}
__device__ __forceinline__ bool csv_is_crlf(uint8_t c) { return c == '\n' || c == '\r'; }

// does byte class `cls` emit a separator from state `s` (prev_term: the byte before is CR / LF, or this is the chunk's first)
__device__ __forceinline__ bool csv_emits(uint32_t s, uint32_t cls, bool prev_term) {
    if (cls == 2) return s != ST_QUO;
    if (cls == 3) return s == ST_UNQ || s == ST_QSEEN || (s == ST_FIELD && !prev_term);
    return false;
}

// the tile's bytes into shared memory (coalesced byte loads; the chunk start has no alignment); returns the thread's
// first byte offset in the tile
__device__ __forceinline__ void csv_load_tile(const uint8_t* __restrict__ chunk, uint64_t n, uint64_t base, uint8_t* s_bytes) {
    for (int k = threadIdx.x; k < CSV_TILE; k += CSV_THREADS) {
        const uint64_t p = base + k;
        s_bytes[k] = p < n ? __ldg(chunk + p) : (uint8_t)0;
    }
    __syncthreads();
}

__device__ __forceinline__ CsvSeg<4> csv_thread_seg(const uint8_t* s_bytes, uint8_t prev, int nb, uint8_t delim) {
    CsvSeg<4> g = csv_seg_identity<4>();
    const int t0 = threadIdx.x * CSV_BPT;
    for (int k = 0; k < nb; ++k) {
        const uint8_t c = s_bytes[t0 + k];
        const uint32_t cls = csv_class(c, delim), nx = csv_next(cls);
        const bool pt = csv_is_crlf(prev);
        uint32_t m = 0;
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const uint32_t cur = (g.map >> (2 * s)) & 3;
            g.c[s] += csv_emits(cur, cls, pt);
            m |= ((nx >> (2 * cur)) & 3) << (2 * s);
        }
        g.map = m;
        prev = c;
    }
    return g;
}

__device__ __forceinline__ CsvSeg<7> csv_thread_seg7(const uint8_t* s_bytes, const uint32_t* s_lut, int nb) {
    CsvSeg<7> g = csv_seg_identity<7>();
    const int t0 = threadIdx.x * CSV_BPT;
    for (int k = 0; k < nb; ++k) {
        const uint32_t t = s_lut[s_bytes[t0 + k]];
        uint32_t m = 0;
#pragma unroll
        for (int s = 0; s < 7; ++s) {
            const uint32_t cur = csv_at<7>(g.map, s);
            g.c[s] += (t >> (G_EMIT + cur)) & 1u;
            m |= csv_at<7>(t, cur) << (3 * s);
        }
        g.map = m;
    }
    return g;
}

// the byte before the thread's first byte; the chunk's first byte counts as following a terminator
__device__ __forceinline__ uint8_t csv_prev_byte(const uint8_t* __restrict__ chunk, uint64_t pos, const uint8_t* s_bytes, int k) {
    if (pos == 0) return '\n';
    return k > 0 ? s_bytes[k - 1] : __ldg(chunk + pos - 1);
}

__device__ __forceinline__ int csv_thread_bytes(uint64_t pos, uint64_t n) {
    return pos >= n ? 0 : (int)(n - pos < (uint64_t)CSV_BPT ? n - pos : (uint64_t)CSV_BPT);
}

// warp inclusive scan of the segments; x becomes the lane's inclusive prefix
template <int NS>
__device__ __forceinline__ CsvSeg<NS> csv_warp_scan(CsvSeg<NS> x) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const CsvSeg<NS> y = csv_shfl_up(x, o);
        if (lane >= o) x = csv_combine(y, x);
    }
    return x;
}

// the general machine's transition words (`lut`, 256 entries) into shared memory; NS == 4 has none
template <int NS>
__device__ __forceinline__ void csv_load_lut(const uint32_t* __restrict__ lut, uint32_t* s_lut) {
    static_assert(CSV_THREADS == 256, "one transition word per thread");
    if (NS != 4) s_lut[threadIdx.x] = __ldg(lut + threadIdx.x);
}

// the thread's segment from its bytes: NS == 4 is the default format's machine, NS == 7 the general one
template <int NS>
__device__ __forceinline__ CsvSeg<NS> csv_thread_segment(const uint8_t* s_bytes, uint8_t prev, int nb, uint8_t delim, const uint32_t* s_lut) {
    if constexpr (NS == 4) return csv_thread_seg(s_bytes, prev, nb, delim);
    else return csv_thread_seg7(s_bytes, s_lut, nb);
}

template <int NS>
__global__ void __launch_bounds__(CSV_THREADS) csv_tok_pass1_kernel(const uint8_t* __restrict__ chunk, uint64_t n, uint8_t delim,
                                                                   const uint32_t* __restrict__ lut, CsvSeg<NS>* __restrict__ tiles) {
    __shared__ uint8_t s_bytes[CSV_TILE];
    __shared__ CsvSeg<NS> s_warp[CSV_THREADS / 32];
    __shared__ uint32_t s_lut[NS == 4 ? 1 : 256];
    const uint64_t base = (uint64_t)blockIdx.x * CSV_TILE;
    csv_load_lut<NS>(lut, s_lut);
    csv_load_tile(chunk, n, base, s_bytes);
    const int k0 = threadIdx.x * CSV_BPT;
    const uint64_t pos = base + k0;
    const uint8_t prev = NS == 4 ? csv_prev_byte(chunk, pos, s_bytes, k0) : 0;  // the general machine has no previous-byte rule
    const CsvSeg<NS> mine = csv_thread_segment<NS>(s_bytes, prev, csv_thread_bytes(pos, n), delim, s_lut);
    const CsvSeg<NS> inc = csv_warp_scan(mine);
    if ((threadIdx.x & 31) == 31) s_warp[threadIdx.x >> 5] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
        CsvSeg<NS> t = s_warp[0];
        for (int w = 1; w < CSV_THREADS / 32; ++w) t = csv_combine(t, s_warp[w]);
        tiles[blockIdx.x] = t;
    }
}

struct CsvInfo {
    unsigned long long err_key;     // min over errors of 2 * separator index (+1: a value error in that field)
    unsigned long long n_seps;      // separators of the chunk (before the virtual terminator of the input's last record)
    unsigned long long last_term;   // 1 + separator index of the last record terminator (0: none)
    unsigned long long n_rec;       // complete records of the chunk
    unsigned long long consumed;    // bytes up to and including the last record terminator
    unsigned long long n_fallback;  // Float64 fields for the host's slow path
    uint32_t end_state, unterminated;
};
struct CsvColInfo {
    unsigned long long nulls;
    unsigned long long vtail, btail;  // the chunk's last 64 validity / Boolean value bits (bit k: row n - 64 + k)
};
struct CsvFallback {
    uint32_t row, col, off, len;
};

// one CTA: the tiles' start states and separator bases (exclusive scan of the segments from state 0, the state a chunk
// starts in: field start after a terminator, or record start)
template <int NS>
__global__ void __launch_bounds__(1024) csv_tok_scan_kernel(const CsvSeg<NS>* __restrict__ tiles, int64_t n_tiles, uint32_t* __restrict__ tile_state,
                                                            uint32_t* __restrict__ tile_base, CsvInfo* __restrict__ info) {
    __shared__ CsvSeg<NS> s[1024];
    const int64_t per = (n_tiles + 1023) / 1024;
    const int64_t lo = (int64_t)threadIdx.x * per, hi = lo + per < n_tiles ? lo + per : n_tiles;
    CsvSeg<NS> m = csv_seg_identity<NS>();
    for (int64_t t = lo; t < hi; ++t) m = csv_combine(m, tiles[t]);
    s[threadIdx.x] = m;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        CsvSeg<NS> y;
        const bool take = (int)threadIdx.x >= o;
        if (take) y = s[threadIdx.x - o];
        __syncthreads();
        if (take) s[threadIdx.x] = csv_combine(y, s[threadIdx.x]);
        __syncthreads();
    }
    uint32_t st = 0, base = 0;
    if (threadIdx.x) {
        const CsvSeg<NS>& p = s[threadIdx.x - 1];
        base = p.c[0];
        st = csv_at<NS>(p.map, 0);
    }
    for (int64_t t = lo; t < hi; ++t) {
        tile_state[t] = st;
        tile_base[t] = base;
        const CsvSeg<NS>& g = tiles[t];
        base += g.c[st];
        st = csv_at<NS>(g.map, st);
    }
    if (threadIdx.x == 1023) {
        info->n_seps = s[1023].c[0];
        info->end_state = csv_at<NS>(s[1023].map, 0);
    }
}

template <int NS>
__global__ void __launch_bounds__(CSV_THREADS) csv_tok_pass2_kernel(const uint8_t* __restrict__ chunk, uint64_t n, uint8_t delim, const uint32_t* __restrict__ lut,
                                                                   uint32_t K, const uint32_t* __restrict__ tile_state,
                                                                   const uint32_t* __restrict__ tile_base, uint32_t* __restrict__ sep,
                                                                   CsvInfo* __restrict__ info) {
    __shared__ uint8_t s_bytes[CSV_TILE];
    __shared__ CsvSeg<NS> s_warp[CSV_THREADS / 32];
    __shared__ uint32_t s_lut[NS == 4 ? 1 : 256];
    const uint64_t base = (uint64_t)blockIdx.x * CSV_TILE;
    csv_load_lut<NS>(lut, s_lut);
    csv_load_tile(chunk, n, base, s_bytes);
    const int k0 = threadIdx.x * CSV_BPT;
    const uint64_t pos = base + k0;
    const uint8_t prev0 = NS == 4 ? csv_prev_byte(chunk, pos, s_bytes, k0) : 0;
    const int nb = csv_thread_bytes(pos, n);
    const CsvSeg<NS> mine = csv_thread_segment<NS>(s_bytes, prev0, nb, delim, s_lut);
    const CsvSeg<NS> inc = csv_warp_scan(mine);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    // true start state and separator index of this thread: tile prefix, then the warps before, then the lanes before
    uint32_t st = tile_state[blockIdx.x], g = tile_base[blockIdx.x];
    for (int w = 0; w < warp; ++w) {
        g += s_warp[w].c[st];
        st = csv_at<NS>(s_warp[w].map, st);
    }
    CsvSeg<NS> ex = csv_shfl_up(inc, 1);
    if (lane > 0) {
        g += ex.c[st];
        st = csv_at<NS>(ex.map, st);
    }
    unsigned long long err = ~0ull, last = 0;
    // a separator at byte `at`: its position, and the field count check (one test per separator)
    auto emit = [&](bool is_term, uint32_t at) {
        sep[g] = at;
        const bool at_end = g % K == K - 1;
        if (is_term) {
            if (!at_end && err == ~0ull) err = 2ull * g;  // too few fields
            last = g + 1;
        } else if (at_end && err == ~0ull) {
            err = 2ull * g;  // too many fields
        }
        ++g;
    };
    if constexpr (NS == 4) {
        uint8_t prev = prev0;
        for (int k = 0; k < nb; ++k) {
            const uint8_t c = s_bytes[k0 + k];
            const uint32_t cls = csv_class(c, delim);
            if (csv_emits(st, cls, csv_is_crlf(prev))) emit(cls == 3, (uint32_t)(pos + k));
            st = (csv_next(cls) >> (2 * st)) & 3;
            prev = c;
        }
    } else {
        for (int k = 0; k < nb; ++k) {
            const uint32_t t = s_lut[s_bytes[k0 + k]];
            if ((t >> (G_EMIT + st)) & 1u) emit((t >> G_TERM) & 1u, (uint32_t)(pos + k));
            st = csv_at<7>(t, st);
        }
    }
    if (err != ~0ull) atomicMin(&info->err_key, err);
    if (last) atomicMax(&info->last_term, last);
}

// the end states after which the input's last record is still open (it gets a virtual terminator) or inside quotes
template <int NS>
__device__ __forceinline__ bool csv_end_open(uint32_t s) { return NS == 4 ? s != ST_FIELD : (s == G_FIELD || s == G_UNQ || s == G_QSEEN); }
template <int NS>
__device__ __forceinline__ bool csv_end_quoted(uint32_t s) { return NS == 4 ? s == ST_QUO : (s == G_QUO || s == G_ESC); }

// one thread: the input's last record without a terminator gets a virtual one at the chunk's end; the complete records
// and the bytes they span. The chunk ends after the terminator of its last complete record (separator n_rec * K - 1), not
// after its last terminator: a terminator past that one closes a record with too few fields, whose error lies beyond the
// complete records, so the next chunk must start with that record and report it.
template <int NS>
__global__ void csv_tok_finish_kernel(uint32_t* __restrict__ sep, uint64_t n, uint32_t K, int is_last, CsvInfo* __restrict__ info) {
    unsigned long long total = info->n_seps, last = info->last_term;
    if (is_last) {
        if (csv_end_quoted<NS>(info->end_state)) {
            info->unterminated = 1;
        } else if (csv_end_open<NS>(info->end_state) || (NS == 4 && total % K != 0)) {
            if (total % K != K - 1) atomicMin(&info->err_key, 2ull * total);
            sep[total] = (uint32_t)n;
            last = ++total;
        }
    }
    info->n_rec = last / K;
    info->last_term = last;
    info->consumed = last >= K ? (unsigned long long)sep[last / K * K - 1] + 1 : 0ull;
    if (info->consumed > n) info->consumed = n;
}

// ---------------------------------------------------------------------------------------------------------------------
// K8b column parsers
// ---------------------------------------------------------------------------------------------------------------------
// field j of record r: [start, end) of the chunk; field 0 skips the CR / LF of blank lines or of a CRLF before it (the
// general format: blank records and comment lines)
template <bool GEN>
__device__ __forceinline__ void csv_field(const uint8_t* __restrict__ chunk, const uint32_t* __restrict__ sep, uint64_t r, uint32_t K, uint32_t j,
                                          const CsvFieldFmt& f, uint32_t* s, uint32_t* e) {
    const uint64_t g = r * K + j;
    *e = sep[g];
    uint32_t a = g ? sep[g - 1] + 1 : 0;
    if (j == 0) {
        if (GEN) a = csv_record_start(chunk, a, *e, f.comment, f.term);
        else
            while (a < *e && csv_is_crlf(chunk[a])) ++a;
    }
    *s = a;
}

struct CsvColArgs {
    uint32_t K, j, first;   // first: records of the chunk to skip (the header)
    char unit;
    CsvFieldFmt fmt;        // the general format (csv_parse_kernel<KIND, true>)
    void* values;           // fixed width: the column's values at its first new row; Boolean: chunk-relative value words
    uint32_t* valid;        // chunk-relative validity words
    CsvColInfo* col;
    // Float64
    CsvFallback* fb;
    uint32_t fb_cap;
    // Utf8
    uint64_t* row_ent;
    unsigned long long* block_bytes;
};

// GEN: the general format's fields, unescaped in place (non-string ones too) and tested against the NULL regex
template <int32_t KIND, bool GEN>
__global__ void __launch_bounds__(CSV_THREADS) csv_parse_kernel(uint8_t* __restrict__ chunk, const uint32_t* __restrict__ sep, CsvInfo* __restrict__ info,
                                                               CsvColArgs a) {
    const int lane = threadIdx.x & 31;
    const uint64_t n_rec = info->n_rec;
    const uint64_t n_out = n_rec > a.first ? n_rec - a.first : 0;
    const uint64_t warps = (uint64_t)gridDim.x * (CSV_THREADS / 32);
    unsigned long long nulls = 0, err = ~0ull;
    for (uint64_t o0 = ((uint64_t)blockIdx.x * (CSV_THREADS / 32) + (threadIdx.x >> 5)) * 32; o0 < n_out; o0 += warps * 32) {
        const uint64_t o = o0 + lane, r = o + a.first;
        const bool in = o < n_out;
        int32_t st = CSV_NULL;
        uint64_t v = 0;
        uint32_t len = 0;
        if (in) {
            uint32_t s, e;
            csv_field<GEN>(chunk, sep, r, a.K, a.j, a.fmt, &s, &e);
            if (KIND == CSV_UTF8) {
                if (GEN) {
                    st = csv_parse_general(KIND, a.unit, chunk + s, e - s, a.fmt, &v, &len);
                } else {
                    len = csv_unescape(chunk + s, e - s, chunk + s);
                    st = len == 0 ? CSV_NULL : len > PQ_STR_MAX_LEN ? CSV_LONG : csv_utf8_valid(chunk + s, len) ? CSV_OK : CSV_BADUTF8;
                }
                if (st != CSV_OK) len = 0;
                a.row_ent[o] = pq_str_ent(s, len);
            } else {
                st = GEN ? csv_parse_general(KIND, a.unit, chunk + s, e - s, a.fmt, &v, &len) : csv_parse_fixed(KIND, a.unit, chunk + s, e - s, &v);
                if (st == CSV_SLOW) {
                    const unsigned long long k = atomicAdd(&info->n_fallback, 1ull);
                    if (k < a.fb_cap) a.fb[k] = CsvFallback{(uint32_t)o, a.j, s, e - s};
                    v = 0;
                    st = CSV_OK;
                }
                if (st != CSV_OK) v = 0;
                if (KIND == CSV_I64 || KIND == CSV_F64 || KIND == CSV_TS) static_cast<uint64_t*>(a.values)[o] = v;
                else if (KIND == CSV_I32 || KIND == CSV_DATE32) static_cast<uint32_t*>(a.values)[o] = (uint32_t)v;
            }
            if (st != CSV_OK && st != CSV_NULL) err = min(err, 2ull * (r * a.K + a.j) + 1);
        }
        const unsigned ok = __ballot_sync(0xffffffffu, st == CSV_OK);
        nulls += __popc(__ballot_sync(0xffffffffu, in && st == CSV_NULL));
        if (KIND == CSV_BOOL) {
            const unsigned bits = __ballot_sync(0xffffffffu, st == CSV_OK && v != 0);
            if (lane == 0) static_cast<uint32_t*>(a.values)[o0 / 32] = bits;
        }
        if (KIND == CSV_UTF8) {
            unsigned long long sum = len;
#pragma unroll
            for (int m = 16; m > 0; m >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, m);
            if (lane == 0 && sum) atomicAdd(a.block_bytes + o0 / PQ_BLOCK_ROWS, sum);
        }
        if (lane == 0) a.valid[o0 / 32] = ok;
    }
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) err = min(err, __shfl_xor_sync(0xffffffffu, err, m));
    if (lane == 0) {
        if (nulls) atomicAdd(&a.col->nulls, nulls);
        if (err != ~0ull) atomicMin(&info->err_key, err);
    }
}

__device__ __forceinline__ unsigned long long csv_last64(const uint32_t* __restrict__ words, uint64_t n) {
    unsigned long long x = 0;
    for (int k = 0; k < 64; ++k) {
        if (n + k < 64) continue;
        const uint64_t row = n + k - 64;
        x |= (unsigned long long)((words[row >> 5] >> (row & 31)) & 1u) << k;
    }
    return x;
}

// one thread per column: the last 64 validity / Boolean value bits (the host mirrors of the columns' partial bytes)
__global__ void csv_tail_kernel(CsvInfo* __restrict__ info, CsvColInfo* __restrict__ cols, const uint32_t* __restrict__ vwords,
                                const uint32_t* __restrict__ bwords, uint64_t stride, uint32_t K, uint32_t first) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= K) return;
    const uint64_t n_rec = info->n_rec, n = n_rec > first ? n_rec - first : 0;
    cols[j].vtail = csv_last64(vwords + j * stride, n);
    cols[j].btail = csv_last64(bwords + j * stride, n);
}

// ---------------------------------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------------------------------
namespace {

struct CsvCol {
    std::string name, fmt;
    int32_t kind = 0, dtype = 0;
    char unit = 0;
    const char* type_name = "";
};

const char* ts_name(char u) {
    return u == 's' ? "Timestamp(Second, None)" : u == 'm' ? "Timestamp(Millisecond, None)" : u == 'u' ? "Timestamp(Microsecond, None)"
                                                                                                  : "Timestamp(Nanosecond, None)";
}

// the Arrow type a format string names (for the refusal message)
std::string arrow_type_of(const std::string& f) {
    static const char* const names[][2] = {{"n", "Null"}, {"b", "Boolean"}, {"c", "Int8"}, {"C", "UInt8"}, {"s", "Int16"}, {"S", "UInt16"},
                                           {"i", "Int32"}, {"I", "UInt32"}, {"l", "Int64"}, {"L", "UInt64"}, {"e", "Float16"}, {"f", "Float32"},
                                           {"g", "Float64"}, {"z", "Binary"}, {"Z", "LargeBinary"}, {"u", "Utf8"}, {"U", "LargeUtf8"},
                                           {"vu", "Utf8View"}, {"vz", "BinaryView"}, {"tdD", "Date32"}, {"tdm", "Date64"}, {"tts", "Time32(Second)"},
                                           {"ttm", "Time32(Millisecond)"}, {"ttu", "Time64(Microsecond)"}, {"ttn", "Time64(Nanosecond)"}};
    for (const auto& n : names)
        if (f == n[0]) return n[1];
    if (f.size() > 4 && f.compare(0, 2, "ts") == 0 && f[3] == ':') {
        const char u = f[2];
        const char* unit = u == 's' ? "Second" : u == 'm' ? "Millisecond" : u == 'u' ? "Microsecond" : "Nanosecond";
        return std::string("Timestamp(") + unit + ", Some(\"" + f.substr(4) + "\"))";
    }
    if (f.compare(0, 2, "d:") == 0) return "Decimal(" + f.substr(2) + ")";
    return "Arrow format '" + f + "'";
}

CsvCol csv_column(const std::string& name, const std::string& f) {
    CsvCol c;
    c.name = name;
    c.fmt = f;
    if (f == "l") c.kind = CSV_I64, c.dtype = TG_INT64, c.type_name = "Int64";
    else if (f == "i") c.kind = CSV_I32, c.dtype = TG_INT32, c.type_name = "Int32";
    else if (f == "g") c.kind = CSV_F64, c.dtype = TG_FLOAT64, c.type_name = "Float64";
    else if (f == "b") c.kind = CSV_BOOL, c.dtype = TG_BOOL, c.type_name = "Boolean";
    else if (f == "u") c.kind = CSV_UTF8, c.dtype = TG_UTF8, c.type_name = "Utf8";
    else if (f == "tdD") c.kind = CSV_DATE32, c.dtype = TG_INT32, c.type_name = "Date32";
    else if (f == "tss:" || f == "tsm:" || f == "tsu:" || f == "tsn:") c.kind = CSV_TS, c.dtype = TG_INT64, c.unit = f[2], c.type_name = ts_name(f[2]);
    else
        throw Error(TG_ERR_UNSUPPORTED, "CSV column '" + name + "': " + arrow_type_of(f) +
                                            " is not supported (Int64, Int32, Float64, Boolean, Utf8, Date32 and naive Timestamp columns are)");
    return c;
}

int64_t env_chunk_bytes() {
    const char* s = getenv("TG_CSV_CHUNK_BYTES");
    const long long v = s ? atoll(s) : 0;
    return v > 0 ? (int64_t)v : (int64_t)256 << 20;
}

// a tg_csv_format with its defaults filled in and checked
struct CsvFormat {
    int32_t delim = ',', quote = '"', esc = -1, comment = -1, term = -1;
    bool header = true;
    std::vector<uint8_t> null_tab;  // csv_null_match's table; empty: no NULL regex
    // the default format runs the 4-state machine and the default field rules; any other the general ones
    bool general() const { return quote != '"' || esc >= 0 || comment >= 0 || term >= 0 || !null_tab.empty(); }
    CsvFieldFmt field(const uint8_t* tab) const { return CsvFieldFmt{quote, esc, comment, term, null_tab.empty() ? nullptr : tab}; }
};

std::string byte_name(int32_t b) {
    char s[8];
    if (b > 32 && b < 127) snprintf(s, sizeof s, "'%c'", (char)b);
    else snprintf(s, sizeof s, "0x%02X", (unsigned)b);
    return s;
}

CsvFormat csv_format(const tg_csv_format* f) {
    if (!f) throw Error(TG_ERR_INVALID_ARG, "CSV: NULL format");
    CsvFormat r;
    const std::pair<const char*, int32_t> in[] = {{"delimiter", f->delimiter}, {"quote", f->quote}, {"escape", f->escape}, {"comment", f->comment},
                                                  {"terminator", f->terminator}};
    for (const auto& x : in)
        if (x.second < -1 || x.second > 255) throw Error(TG_ERR_INVALID_ARG, std::string("CSV: the ") + x.first + " must be a byte (0..255) or -1");
    if (f->delimiter >= 0) r.delim = f->delimiter;
    if (f->quote >= 0) r.quote = f->quote;
    r.esc = f->escape;
    r.comment = f->comment;
    r.term = f->terminator;
    r.header = f->has_header != 0;
    // the special bytes are pairwise distinct (the default terminator is both CR and LF)
    std::vector<std::pair<std::string, int32_t>> sp = {{"delimiter", r.delim}, {"quote", r.quote}, {"escape", r.esc}, {"comment", r.comment}};
    if (r.term >= 0) sp.push_back({"terminator", r.term});
    else sp.insert(sp.end(), {{"terminator (LF)", '\n'}, {"terminator (CR)", '\r'}});
    for (size_t i = 0; i < sp.size(); ++i)
        for (size_t j = i + 1; j < sp.size(); ++j)
            if (sp[i].second >= 0 && sp[i].second == sp[j].second)
                throw Error(TG_ERR_INVALID_ARG, "CSV: the " + sp[i].first + " and the " + sp[j].first + " are the same byte " + byte_name(sp[i].second));
    if (f->null_regex) {
        Dfa d;
        try {
            d = compile_regex(f->null_regex, false);
        } catch (Error& e) {  // a syntax error is the caller's argument; a construct the DFA compiler refuses stays unsupported
            throw Error(e.code == TG_ERR_UNSUPPORTED ? TG_ERR_UNSUPPORTED : TG_ERR_INVALID_ARG, "CSV: NULL regex: " + e.msg);
        }
        const uint32_t nc = d.n_classes, row = nc + 1;
        r.null_tab.assign(16 + 256 + (size_t)d.n_states * row * 2, 0);
        const uint32_t hdr[2] = {nc, d.start};
        memcpy(r.null_tab.data(), hdr, 8);
        memcpy(r.null_tab.data() + 16, d.class_of, 256);
        uint16_t* rows = reinterpret_cast<uint16_t*>(r.null_tab.data() + 16 + 256);
        for (uint32_t s = 0; s < d.n_states; ++s) {
            for (uint32_t c = 0; c < nc; ++c) rows[(size_t)s * row + c] = d.next[(size_t)s * nc + c];
            rows[(size_t)s * row + nc] = d.accept_end[s];
        }
    }
    return r;
}

// the general machine's transition word of every byte value (see G_REC)
std::vector<uint32_t> csv_machine(const CsvFormat& f) {
    std::vector<uint32_t> lut(256);
    for (int b = 0; b < 256; ++b) {
        const bool quote = b == f.quote, delim = b == f.delim, esc = b == f.esc, comment = b == f.comment;
        const bool term = f.term >= 0 ? b == f.term : (b == '\n' || b == '\r');
        uint32_t w = term ? 1u << G_TERM : 0u;
        for (uint32_t s = 0; s < 7; ++s) {
            uint32_t nx;
            bool emit = false;
            switch (s) {
                case G_REC:
                case G_FIELD:
                    nx = quote ? G_QUO : delim ? G_FIELD : term ? G_REC : (comment && s == G_REC) ? G_CMT : G_UNQ;
                    emit = delim || (term && s == G_FIELD);
                    break;
                case G_UNQ:
                case G_QSEEN:
                    nx = quote ? (s == G_QSEEN ? G_QUO : G_UNQ) : delim ? G_FIELD : term ? G_REC : G_UNQ;
                    emit = delim || term;
                    break;
                case G_QUO: nx = quote ? G_QSEEN : esc ? G_ESC : G_QUO; break;
                case G_ESC: nx = G_QUO; break;
                default: nx = term ? G_REC : G_CMT; break;  // G_CMT
            }
            w |= nx << (3 * s);
            if (emit) w |= 1u << (G_EMIT + s);
        }
        lut[b] = w;
    }
    return lut;
}

// 1-based line of byte `pos` of the n bytes: lines end at the terminator (the default: LF, CRLF or a lone CR)
int64_t line_of(const uint8_t* p, int64_t n, int64_t pos, int32_t term) {
    int64_t line = 1;
    for (int64_t i = 0; i < pos; ++i)
        if (term >= 0 ? p[i] == term : (p[i] == '\n' || (p[i] == '\r' && !(i + 1 < n && p[i + 1] == '\n')))) ++line;
    return line;
}

std::string shown(const uint8_t* p, uint32_t n) {
    std::string s((const char*)p, std::min<uint32_t>(n, 64));
    if (n > 64) s += "...";
    return s;
}

// Float64 through strtod after the device's grammar check (or when it could not check: a too-long list)
// (gen: the general format's field rules, with the host copy of the NULL regex's table)
int32_t csv_f64_slow(const uint8_t* p, uint32_t n, uint64_t* bits, const CsvFieldFmt* gen = nullptr) {
    std::string s((const char*)p, n);
    uint32_t m = 0;
    const int32_t st = gen ? csv_parse_general(CSV_F64, 0, (uint8_t*)&s[0], n, *gen, bits, &m) : csv_parse_fixed(CSV_F64, 0, p, n, bits);
    if (st != CSV_SLOW) return st;
    s.resize(gen ? m : csv_unescape(p, n, (uint8_t*)&s[0]));
    const double d = strtod(s.c_str(), nullptr);
    memcpy(bits, &d, 8);
    return CSV_OK;
}

// device work area of one call, sized for chunks of up to `cap` bytes
struct CsvWork {
    uint8_t* p = nullptr;
    size_t bytes = 0;
    uint64_t cap = 0, bound = 0, words = 0, blocks = 0;
    void* tiles;                         // CsvSeg<4> or CsvSeg<7> per tile
    uint32_t *tile_state, *tile_base, *sep, *vwords, *bwords;
    CsvInfo* info;
    CsvColInfo* cols;
    CsvFallback* fb;
    uint64_t* row_ent;                   // [n utf8 columns][bound]
    unsigned long long *block_bytes, *block_base;  // [n utf8 columns][blocks + 1]
    PqBlock* pq_blocks;                  // [blocks]
};
constexpr uint32_t CSV_FB_CAP = 1u << 16;

void work_alloc(Engine& e, CsvWork& w, uint64_t cap, uint32_t K, uint32_t n_utf8) {
    w.cap = cap;
    w.bound = cap / K + 2;
    w.words = (w.bound + 31) / 32 + 2;
    w.blocks = (w.bound + PQ_BLOCK_ROWS - 1) / PQ_BLOCK_ROWS + 1;
    const uint64_t n_tiles = (cap + CSV_TILE - 1) / CSV_TILE + 1;
    const size_t sz[] = {r16(n_tiles * sizeof(CsvSeg<7>)), r16(n_tiles * 4), r16(n_tiles * 4), r16((cap + 2) * 4), r16(K * w.words * 4), r16(K * w.words * 4),
                         r16(sizeof(CsvInfo)), r16(K * sizeof(CsvColInfo)), r16(CSV_FB_CAP * sizeof(CsvFallback)), r16(n_utf8 * w.bound * 8),
                         r16(n_utf8 * (w.blocks + 1) * 8), r16(n_utf8 * (w.blocks + 1) * 8), r16(w.blocks * sizeof(PqBlock))};
    size_t total = 0;
    for (size_t s : sz) total += s;
    w.p = e.dev_alloc(total);
    w.bytes = total;
    uint8_t* q = w.p;
    auto take = [&](int i) {
        uint8_t* r = q;
        q += sz[i];
        return r;
    };
    w.tiles = take(0);
    w.tile_state = (uint32_t*)take(1);
    w.tile_base = (uint32_t*)take(2);
    w.sep = (uint32_t*)take(3);
    w.vwords = (uint32_t*)take(4);
    w.bwords = (uint32_t*)take(5);
    w.info = (CsvInfo*)take(6);
    w.cols = (CsvColInfo*)take(7);
    w.fb = (CsvFallback*)take(8);
    w.row_ent = (uint64_t*)take(9);
    w.block_bytes = (unsigned long long*)take(10);
    w.block_base = (unsigned long long*)take(11);
    w.pq_blocks = (PqBlock*)take(12);
}

struct CsvEvents {
    cudaEvent_t up_done[2] = {}, buf_free[2] = {};
    CsvEvents() {
        for (int i = 0; i < 2; ++i) {
            TG_CUDA(cudaEventCreateWithFlags(&up_done[i], cudaEventDisableTiming));
            TG_CUDA(cudaEventCreateWithFlags(&buf_free[i], cudaEventDisableTiming));
        }
    }
    ~CsvEvents() {
        for (int i = 0; i < 2; ++i) {
            if (up_done[i]) cudaEventDestroy(up_done[i]);
            if (buf_free[i]) cudaEventDestroy(buf_free[i]);
        }
    }
};

}  // namespace

// the value parser of the device path for one field (the raw field: quoted or not); host-only
void csv_parse_value(const std::string& fmt, const uint8_t* p, int64_t n, void* out, int32_t* is_null) {
    const CsvCol c = csv_column("value", fmt);
    if (n < 0 || (!p && n > 0)) throw Error(TG_ERR_INVALID_ARG, "NULL field");
    if (n > (int64_t)0xFFFFFFFFll) throw Error(TG_ERR_UNSUPPORTED, "a field of 4 GiB or more");
    const uint32_t m = (uint32_t)n;
    if (is_null) *is_null = 0;
    if (c.kind == CSV_UTF8) {
        std::vector<uint8_t> tmp(m + 1);
        const uint32_t len = csv_unescape(p, m, tmp.data());
        if (len == 0) {
            if (is_null) *is_null = 1;
        } else if (!csv_utf8_valid(tmp.data(), len)) {
            throw Error(TG_ERR_INVALID_ARG, "invalid UTF-8");
        }
        if (out) *(int64_t*)out = len;
        return;
    }
    uint64_t v = 0;
    const int32_t st = c.kind == CSV_F64 ? csv_f64_slow(p, m, &v) : csv_parse_fixed(c.kind, c.unit, p, m, &v);
    if (st == CSV_NULL) {
        if (is_null) *is_null = 1;
        v = 0;
    } else if (st == CSV_RANGE) {
        throw Error(TG_ERR_INVALID_ARG, "'" + shown(p, m) + "' is out of range for " + c.type_name);
    } else if (st != CSV_OK) {
        throw Error(TG_ERR_INVALID_ARG, "cannot parse '" + shown(p, m) + "' as " + c.type_name);
    }
    if (!out) return;
    if (c.kind == CSV_I32 || c.kind == CSV_DATE32) *(int32_t*)out = (int32_t)v;
    else if (c.kind == CSV_BOOL) *(uint8_t*)out = (uint8_t)v;
    else memcpy(out, &v, 8);
}

// the general machine run on the host one byte at a time, with the device's field rules (tg_csv_split_host)
void csv_split_host(const tg_csv_format* format, const uint8_t* p, int64_t n, uint8_t* values, int64_t* value_ends, uint8_t* is_null,
                    int64_t* record_fields, int64_t* record_lines, int64_t* n_fields, int64_t* n_records) {
    const CsvFormat f = csv_format(format);
    if (n < 0 || (!p && n > 0)) throw Error(TG_ERR_INVALID_ARG, "CSV: NULL bytes");
    if (n >= 0xFFFFFFF0ll) throw Error(TG_ERR_UNSUPPORTED, "CSV: 4 GiB or more");
    if (n > 0 && (!values || !value_ends || !is_null || !record_fields || !record_lines)) throw Error(TG_ERR_INVALID_ARG, "NULL output");
    const std::vector<uint32_t> lut = csv_machine(f);
    const CsvFieldFmt ff = f.field(f.null_tab.data());
    int64_t nf = 0, nr = 0, out = 0, rec_first = 0, rec_line = 1, line = 1, lp = 0;
    auto line_at = [&](int64_t pos) {  // incremental line_of
        for (; lp < pos; ++lp)
            if (f.term >= 0 ? p[lp] == f.term : (p[lp] == '\n' || (p[lp] == '\r' && !(lp + 1 < n && p[lp + 1] == '\n')))) ++line;
        return line;
    };
    auto field = [&](uint32_t a, uint32_t e, bool ends_record) {
        if (nf == rec_first) {
            a = csv_record_start(p, a, e, f.comment, f.term);
            rec_line = line_at(a);
        }
        memcpy(values + out, p + a, e - a);
        const uint32_t m = csv_unescape(values + out, e - a, values + out, f.quote, f.esc);
        is_null[nf] = ff.null_tab ? csv_null_match(ff.null_tab, values + out, m) : m == 0;
        out += m;
        value_ends[nf++] = out;
        if (ends_record) {
            record_fields[nr] = nf - rec_first;
            record_lines[nr++] = rec_line;
            rec_first = nf;
        }
    };
    uint32_t st = G_REC, fs = 0;
    for (uint32_t i = 0; i < (uint32_t)n; ++i) {
        const uint32_t t = lut[p[i]];
        if ((t >> (G_EMIT + st)) & 1u) {
            field(fs, i, (t >> G_TERM) & 1u);
            fs = i + 1;
        }
        st = (t >> (3 * st)) & 7u;
    }
    if (st == G_QUO || st == G_ESC) {
        const int64_t l = nf == rec_first ? line_at(csv_record_start(p, fs, (uint32_t)n, f.comment, f.term)) : rec_line;
        throw Error(TG_ERR_INVALID_ARG, "CSV line " + std::to_string(l) + ": unterminated quote at the end of the input");
    }
    if (st == G_FIELD || st == G_UNQ || st == G_QSEEN) field(fs, (uint32_t)n, true);
    if (n_fields) *n_fields = nf;
    if (n_records) *n_records = nr;
}

void table_append_csv(Table& t, const std::vector<std::string>& names, const std::vector<std::string>& fmts, const uint8_t* bytes, int64_t n_bytes,
                      const tg_csv_format* format, int64_t* rows_out) {
    AppendTxn txn(t);
    Engine& e = txn.e;
    const uint32_t K = (uint32_t)names.size();
    if (K == 0) throw Error(TG_ERR_INVALID_ARG, "CSV: no columns");
    if (n_bytes < 0 || (!bytes && n_bytes > 0)) throw Error(TG_ERR_INVALID_ARG, "CSV: NULL bytes");
    const CsvFormat fmt = csv_format(format);
    const bool gen = fmt.general();
    std::vector<CsvCol> cols;
    uint32_t n_utf8 = 0;
    for (uint32_t j = 0; j < K; ++j) {
        for (uint32_t i = 0; i < j; ++i)
            if (names[i] == names[j]) throw Error(TG_ERR_INVALID_ARG, "CSV: column '" + names[j] + "' is listed twice");
        cols.push_back(csv_column(names[j], fmts[j]));
        n_utf8 += cols.back().kind == CSV_UTF8;
    }
    // a column keeps one delivered type (checked before anything is appended)
    for (const CsvCol& c : cols) {
        Column* have = t.find(c.name);
        if (!have) continue;
        const bool temporal = c.kind == CSV_DATE32 || c.kind == CSV_TS;
        const char* src = c.kind == CSV_TS ? "Timestamp" : "Date32";
        const bool same = have->dtype == c.dtype && (temporal ? have->src_type && strcmp(have->src_type, src) == 0 && have->temporal &&
                                                                    have->temporal_unit == (c.kind == CSV_TS ? c.unit : 'D')
                                                              : have->src_type == nullptr);
        if (!same) throw Error(TG_ERR_TYPE_MISMATCH, "column '" + c.name + "' was registered with a different type than " + c.type_name);
    }
    CsvWork w;
    uint8_t* buf[2] = {nullptr, nullptr};
    size_t buf_bytes = 0;
    uint8_t* aux = nullptr;  // the general format: the machine's transition words, then the NULL regex's table
    size_t aux_bytes = 0;
    // the Utf8 tails read the staging buffers asynchronously: released at the next sync_copies, after a failed call too (the
    // transaction has then waited for the streams)
    auto release_staging = [&] {
        const std::pair<uint8_t*, size_t> blocks[] = {{buf[0], buf_bytes}, {buf[1], buf_bytes}, {w.p, w.bytes}, {aux, aux_bytes}};
        for (const auto& b : blocks)
            if (b.first) e.deferred_free.push_back(b);
    };
    try {
        std::vector<Column*> dcols;
        for (const CsvCol& c : cols) {
            Column& col = txn.column(c.name, c.dtype);
            if (c.kind == CSV_DATE32 || c.kind == CSV_TS) declare_arrow_type(col, c.fmt);
            dcols.push_back(&col);
        }
        int64_t rows = 0;
        if (n_bytes > 0) {
            e.ensure_side_streams();
            cudaStream_t up = e.side[0];
            CsvEvents ev;
            const uint64_t L = (uint64_t)env_chunk_bytes();
            uint64_t C = L;  // room in front of a window for the record the previous chunk cut off
            auto alloc_bufs = [&]() {
                buf_bytes = C + L + 16;
                buf[0] = e.dev_alloc(buf_bytes);
                buf[1] = e.dev_alloc(buf_bytes);
            };
            alloc_bufs();
            work_alloc(e, w, C + L, K, n_utf8);
            if (gen) {
                const std::vector<uint32_t> lut = csv_machine(fmt);
                aux_bytes = 1024 + r16(fmt.null_tab.size());
                aux = e.dev_alloc(aux_bytes);
                e.h2d(aux, lut.data(), 1024);
                e.h2d(aux + 1024, fmt.null_tab.data(), fmt.null_tab.size());
            }
            const uint32_t* d_lut = reinterpret_cast<const uint32_t*>(aux);
            const CsvFieldFmt dfmt = fmt.field(aux ? aux + 1024 : nullptr), hfmt = fmt.field(fmt.null_tab.data());
            const uint64_t n_windows = ((uint64_t)n_bytes + L - 1) / L;
            auto win_len = [&](uint64_t k) { return std::min<uint64_t>(L, (uint64_t)n_bytes - k * L); };
            auto upload = [&](uint64_t k) {
                const int b = (int)(k & 1);
                TG_CUDA(cudaStreamWaitEvent(up, ev.buf_free[b], 0));
                e.h2d(buf[b] + C, bytes + k * L, win_len(k), up);
                TG_CUDA(cudaEventRecord(ev.up_done[b], up));
            };
            TG_CUDA(cudaEventRecord(ev.buf_free[0], e.copy_stream));
            TG_CUDA(cudaEventRecord(ev.buf_free[1], e.copy_stream));
            upload(0);
            uint64_t carry = 0;
            const uint8_t* carry_src = nullptr;
            bool header = fmt.header;
            for (uint64_t k = 0; k < n_windows; ++k) {
                const int b = (int)(k & 1);
                const bool is_last = k + 1 == n_windows;
                TG_CUDA(cudaStreamWaitEvent(e.copy_stream, ev.up_done[b], 0));
                if (carry + L >= 0xFFFFFFF0ull) throw Error(TG_ERR_UNSUPPORTED, "CSV: a record of 4 GiB or more");
                if (carry > C) {  // a record longer than the room: grow the buffers (and the work area) and move both parts over
                    TG_CUDA(cudaStreamSynchronize(up));
                    TG_CUDA(cudaStreamSynchronize(e.copy_stream));
                    const uint64_t C2 = std::max<uint64_t>(2 * C, carry + L);
                    uint8_t* old[2] = {buf[0], buf[1]};
                    const size_t old_bytes = buf_bytes;
                    const uint64_t C_old = C;
                    C = C2;
                    alloc_bufs();
                    TG_CUDA(cudaMemcpyAsync(buf[b] + C - carry, carry_src, carry, cudaMemcpyDeviceToDevice, e.copy_stream));
                    TG_CUDA(cudaMemcpyAsync(buf[b] + C, old[b] + C_old, win_len(k), cudaMemcpyDeviceToDevice, e.copy_stream));
                    TG_CUDA(cudaStreamSynchronize(e.copy_stream));
                    e.dev_free(old[0], old_bytes);
                    e.dev_free(old[1], old_bytes);
                    e.dev_free(w.p, w.bytes);
                    work_alloc(e, w, C + L, K, n_utf8);
                } else if (carry) {
                    TG_CUDA(cudaMemcpyAsync(buf[b] + C - carry, carry_src, carry, cudaMemcpyDeviceToDevice, e.copy_stream));
                }
                TG_CUDA(cudaEventRecord(ev.buf_free[b ^ 1], e.copy_stream));
                uint8_t* chunk = buf[b] + C - carry;
                const uint64_t len = carry + win_len(k);
                const int64_t file_off = (int64_t)(k * L) - (int64_t)carry;
                const uint32_t first = header ? 1 : 0;
                // ---- K8a
                TG_CUDA(cudaMemsetAsync(w.info, 0, sizeof(CsvInfo), e.copy_stream));
                TG_CUDA(cudaMemsetAsync(&w.info->err_key, 0xFF, 8, e.copy_stream));
                TG_CUDA(cudaMemsetAsync(w.cols, 0, K * sizeof(CsvColInfo), e.copy_stream));
                const uint64_t n_tiles = (len + CSV_TILE - 1) / CSV_TILE;
                const uint8_t delim = (uint8_t)fmt.delim;
                if (gen) {
                    CsvSeg<7>* tiles = static_cast<CsvSeg<7>*>(w.tiles);
                    csv_tok_pass1_kernel<7><<<(unsigned)n_tiles, CSV_THREADS, 0, e.copy_stream>>>(chunk, len, delim, d_lut, tiles);
                    csv_tok_scan_kernel<7><<<1, 1024, 0, e.copy_stream>>>(tiles, (int64_t)n_tiles, w.tile_state, w.tile_base, w.info);
                    csv_tok_pass2_kernel<7><<<(unsigned)n_tiles, CSV_THREADS, 0, e.copy_stream>>>(chunk, len, delim, d_lut, K, w.tile_state, w.tile_base,
                                                                                                 w.sep, w.info);
                    csv_tok_finish_kernel<7><<<1, 1, 0, e.copy_stream>>>(w.sep, len, K, is_last ? 1 : 0, w.info);
                } else {
                    CsvSeg<4>* tiles = static_cast<CsvSeg<4>*>(w.tiles);
                    csv_tok_pass1_kernel<4><<<(unsigned)n_tiles, CSV_THREADS, 0, e.copy_stream>>>(chunk, len, delim, nullptr, tiles);
                    csv_tok_scan_kernel<4><<<1, 1024, 0, e.copy_stream>>>(tiles, (int64_t)n_tiles, w.tile_state, w.tile_base, w.info);
                    csv_tok_pass2_kernel<4><<<(unsigned)n_tiles, CSV_THREADS, 0, e.copy_stream>>>(chunk, len, delim, nullptr, K, w.tile_state, w.tile_base,
                                                                                                 w.sep, w.info);
                    csv_tok_finish_kernel<4><<<1, 1, 0, e.copy_stream>>>(w.sep, len, K, is_last ? 1 : 0, w.info);
                }
                TG_CUDA(cudaGetLastError());
                e.launches += 4;
                // ---- K8b: every column into its reserved tail
                const uint64_t bound = len / K + 2;
                const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>((bound + CSV_THREADS - 1) / CSV_THREADS, (uint64_t)e.sm_count * 8));
                uint32_t u = 0;
                for (uint32_t j = 0; j < K; ++j) {
                    Column& c = *dcols[j];
                    const int64_t have = c.n_rows;
                    CsvColArgs a{};
                    a.K = K;
                    a.j = j;
                    a.first = first;
                    const int32_t kind = cols[j].kind;
                    a.unit = cols[j].unit;
                    a.fmt = dfmt;
                    a.valid = w.vwords + j * w.words;
                    a.col = w.cols + j;
                    a.fb = w.fb;
                    a.fb_cap = CSV_FB_CAP;
                    if (kind == CSV_BOOL) {
                        a.values = w.bwords + j * w.words;
                    } else if (kind == CSV_UTF8) {
                        a.row_ent = w.row_ent + (uint64_t)u * w.bound;
                        a.block_bytes = w.block_bytes + (uint64_t)u * (w.blocks + 1);
                        TG_CUDA(cudaMemsetAsync(a.block_bytes, 0, (w.blocks + 1) * 8, e.copy_stream));
                        ++u;
                    } else {
                        const size_t wb = (size_t)c.elem_bytes();
                        e.dev_reserve(c.values, (size_t)(have + (int64_t)bound) * wb, (size_t)have * wb);
                        a.values = c.values.p + (size_t)have * wb;
                    }
                    using Kern = void (*)(uint8_t*, const uint32_t*, CsvInfo*, CsvColArgs);
                    static const Kern kernels[2][7] = {
                        {csv_parse_kernel<CSV_I64, false>, csv_parse_kernel<CSV_I32, false>, csv_parse_kernel<CSV_F64, false>, csv_parse_kernel<CSV_BOOL, false>,
                         csv_parse_kernel<CSV_UTF8, false>, csv_parse_kernel<CSV_DATE32, false>, csv_parse_kernel<CSV_TS, false>},
                        {csv_parse_kernel<CSV_I64, true>, csv_parse_kernel<CSV_I32, true>, csv_parse_kernel<CSV_F64, true>, csv_parse_kernel<CSV_BOOL, true>,
                         csv_parse_kernel<CSV_UTF8, true>, csv_parse_kernel<CSV_DATE32, true>, csv_parse_kernel<CSV_TS, true>}};
                    kernels[gen][kind]<<<grid, CSV_THREADS, 0, e.copy_stream>>>(chunk, w.sep, w.info, a);
                    TG_CUDA(cudaGetLastError());
                    e.launches += 1;
                }
                csv_tail_kernel<<<(K + 127) / 128, 128, 0, e.copy_stream>>>(w.info, w.cols, w.vwords, w.bwords, w.words, K, first);
                TG_CUDA(cudaGetLastError());
                e.launches += 1;
                // ---- the chunk's one read-back: info, column records, and the head values of columns without a pivot yet
                const uint64_t head = std::min<uint64_t>(bound, 65536);
                std::vector<uint32_t> pivot_cols;
                for (uint32_t j = 0; j < K; ++j)
                    if (!dcols[j]->pivot_set && (dcols[j]->dtype == TG_INT64 || dcols[j]->dtype == TG_FLOAT64)) pivot_cols.push_back(j);
                const size_t info_b = r16(sizeof(CsvInfo) + K * sizeof(CsvColInfo)), head_b = head * 8 + r16((head + 31) / 32 * 4);
                uint8_t* h = e.host_scratch(info_b + pivot_cols.size() * head_b);
                TG_CUDA(cudaMemcpyAsync(h, w.info, sizeof(CsvInfo), cudaMemcpyDeviceToHost, e.copy_stream));
                TG_CUDA(cudaMemcpyAsync(h + sizeof(CsvInfo), w.cols, K * sizeof(CsvColInfo), cudaMemcpyDeviceToHost, e.copy_stream));
                for (size_t i = 0; i < pivot_cols.size(); ++i) {
                    const uint32_t j = pivot_cols[i];
                    uint8_t* hp = h + info_b + i * head_b;
                    TG_CUDA(cudaMemcpyAsync(hp, dcols[j]->values.p + (size_t)dcols[j]->n_rows * 8, head * 8, cudaMemcpyDeviceToHost, e.copy_stream));
                    TG_CUDA(cudaMemcpyAsync(hp + head * 8, w.vwords + j * w.words, (head + 31) / 32 * 4, cudaMemcpyDeviceToHost, e.copy_stream));
                }
                if (!is_last) upload(k + 1);  // the next window's host copy runs while the kernels above do
                TG_CUDA(cudaStreamSynchronize(e.copy_stream));
                CsvInfo info;
                memcpy(&info, h, sizeof(CsvInfo));
                std::vector<CsvColInfo> ci(K);
                memcpy(ci.data(), h + sizeof(CsvInfo), K * sizeof(CsvColInfo));
                if (!is_last && info.n_rec == 0) {  // no record ends in this chunk: it becomes the next chunk's front part
                    carry = len;
                    carry_src = chunk;
                    continue;
                }
                const uint64_t n_out = info.n_rec > first ? info.n_rec - first : 0;
                const uint8_t* hchunk = bytes + file_off;
                // ---- Float64 fields the device could not decide: strtod on the host, patched into place
                unsigned long long err_key = info.err_key;
                const unsigned long long cut = is_last ? ~0ull : 2ull * info.n_rec * K;  // later errors belong to the cut-off record
                std::vector<uint64_t> patches;  // (outlives its queued copies)
                if (info.n_fallback) {
                    // a patched value also replaces the read-back head value the pivot is taken from
                    auto slow = [&](uint64_t o, uint32_t j, uint32_t off, uint32_t flen, uint64_t* bits) {
                        const int32_t st = csv_f64_slow(hchunk + off, flen, bits, gen ? &hfmt : nullptr);
                        if (st != CSV_OK && st != CSV_NULL) {
                            err_key = std::min<unsigned long long>(err_key, 2ull * ((o + first) * (uint64_t)K + j) + 1);
                            return false;
                        }
                        if (st == CSV_OK && o < head)
                            for (size_t i = 0; i < pivot_cols.size(); ++i)
                                if (pivot_cols[i] == j) reinterpret_cast<uint64_t*>(h + info_b + i * head_b)[o] = *bits;
                        return st == CSV_OK;
                    };
                    if (info.n_fallback <= CSV_FB_CAP) {
                        std::vector<CsvFallback> fb(info.n_fallback);
                        TG_CUDA(cudaMemcpy(fb.data(), w.fb, fb.size() * sizeof(CsvFallback), cudaMemcpyDeviceToHost));
                        patches.resize(fb.size());
                        for (size_t i = 0; i < fb.size(); ++i) {
                            const CsvFallback& f = fb[i];
                            if (f.row < n_out && slow(f.row, f.col, f.off, f.len, &patches[i]))
                                TG_CUDA(cudaMemcpyAsync(dcols[f.col]->values.p + (size_t)(dcols[f.col]->n_rows + f.row) * 8, &patches[i], 8,
                                                        cudaMemcpyHostToDevice, e.copy_stream));
                        }
                    } else {  // the list overflowed: every Float64 field of the chunk goes through the host, one copy per column
                        std::vector<uint32_t> sep(info.n_rec * K);
                        TG_CUDA(cudaMemcpy(sep.data(), w.sep, sep.size() * 4, cudaMemcpyDeviceToHost));
                        for (uint32_t j = 0; j < K; ++j) {
                            if (cols[j].kind != CSV_F64) continue;
                            patches.assign(n_out, 0);  // NULL rows hold 0, as the kernel writes them
                            for (uint64_t o = 0; o < n_out; ++o) {
                                const uint64_t gi = (o + first) * K + j;
                                uint32_t fs = gi ? sep[gi - 1] + 1 : 0;
                                const uint32_t fe = sep[gi];
                                if (j == 0) fs = csv_record_start(hchunk, fs, fe, fmt.comment, fmt.term);
                                if (fe > fs || gen) slow(o, j, fs, fe - fs, &patches[o]);
                            }
                            e.h2d(dcols[j]->values.p + (size_t)dcols[j]->n_rows * 8, patches.data(), n_out * 8);
                        }
                    }
                }
                // ---- the first error, with the line its record starts on and the column
                const bool unterminated = is_last && info.unterminated;
                if ((err_key != ~0ull && err_key < cut) || unterminated) {
                    const uint64_t gq = info.n_seps;  // an unterminated quote: the field after the last separator
                    const uint64_t gi = unterminated && (err_key == ~0ull || err_key >= 2 * gq) ? gq : err_key / 2;
                    const bool is_value = !(unterminated && gi == gq) && (err_key & 1);
                    const uint64_t r = gi / K;
                    const uint32_t j = (uint32_t)(gi % K);
                    // separators [rK - 1, gi] of the chunk (an unterminated quote: only the one before its record)
                    const bool quote_err = unterminated && gi == gq;
                    const uint64_t lo = r * K ? r * K - 1 : 0, hi = quote_err ? lo : gi;
                    std::vector<uint32_t> sp(hi - lo + 1, 0);
                    if (!quote_err || r * K) TG_CUDA(cudaMemcpy(sp.data(), w.sep + lo, sp.size() * 4, cudaMemcpyDeviceToHost));
                    auto sep_at = [&](uint64_t x) -> uint64_t { return sp[x - lo]; };
                    uint64_t rs = r * K ? sep_at(r * K - 1) + 1 : 0;
                    rs = csv_record_start(hchunk, (uint32_t)rs, (uint32_t)len, fmt.comment, fmt.term);
                    const std::string where = "CSV line " + std::to_string(line_of(bytes, n_bytes, file_off + (int64_t)rs, fmt.term)) + ", column '" + cols[j].name + "': ";
                    if (quote_err) throw Error(TG_ERR_INVALID_ARG, where + "unterminated quote at the end of the input");
                    const uint64_t fe = sep_at(gi);
                    if (!is_value) {
                        const bool term = fe >= len || csv_is_term(hchunk[fe], fmt.term);
                        const std::string line = "CSV line " + std::to_string(line_of(bytes, n_bytes, file_off + (int64_t)rs, fmt.term));
                        if (term)  // the record ends after field j: column j + 1 is missing
                            throw Error(TG_ERR_INVALID_ARG, line + ", column '" + cols[j + 1].name + "': missing: the record has " + std::to_string(j + 1) +
                                                                " fields, the schema " + std::to_string(K));
                        throw Error(TG_ERR_INVALID_ARG, where + "followed by an extra field: the record has more than the schema's " + std::to_string(K) + " fields");
                    }
                    uint64_t fs = j ? sep_at(gi - 1) + 1 : rs;
                    const uint32_t fn = (uint32_t)(fe - fs);
                    if (cols[j].kind == CSV_UTF8) {
                        std::vector<uint8_t> tmp(fn + 1);
                        const uint32_t ulen = csv_unescape(hchunk + fs, fn, tmp.data(), fmt.quote, fmt.esc);
                        if (ulen > PQ_STR_MAX_LEN) throw Error(TG_ERR_UNSUPPORTED, where + "string value of 16 MiB or more");
                        throw Error(TG_ERR_INVALID_ARG, where + "invalid UTF-8");
                    }
                    uint64_t v;
                    std::vector<uint8_t> tmp(hchunk + fs, hchunk + fs + fn);
                    uint32_t ulen;
                    const int32_t st = gen ? csv_parse_general(cols[j].kind, cols[j].unit, tmp.data(), fn, hfmt, &v, &ulen)
                                           : csv_parse_fixed(cols[j].kind, cols[j].unit, hchunk + fs, fn, &v);
                    if (st == CSV_RANGE) throw Error(TG_ERR_INVALID_ARG, where + "'" + shown(hchunk + fs, fn) + "' is out of range for " + cols[j].type_name);
                    throw Error(TG_ERR_INVALID_ARG, where + "cannot parse '" + shown(hchunk + fs, fn) + "' as " + cols[j].type_name);
                }
                // ---- commit the chunk's rows (pivots first: the commit's own copies may reuse the pinned scratch)
                if (n_out > 0) {
                    for (size_t i = 0; i < pivot_cols.size(); ++i) {
                        Column& c = *dcols[pivot_cols[i]];
                        const uint8_t* hp = h + info_b + i * head_b;
                        set_pivot_host(c, c.dtype, (int64_t)std::min<uint64_t>(n_out, head), hp, hp + head * 8, 0);
                    }
                    u = 0;
                    for (uint32_t j = 0; j < K; ++j) {
                        Column& c = *dcols[j];
                        const int64_t have = c.n_rows;
                        const uint32_t* vw = w.vwords + j * w.words;
                        append_validity_device(e, c, have, vw, (int64_t)n_out, (int64_t)ci[j].nulls, ci[j].vtail);
                        if (cols[j].kind == CSV_UTF8) {
                            const uint64_t nb = (n_out + PQ_BLOCK_ROWS - 1) / PQ_BLOCK_ROWS;
                            std::vector<PqBlock> blocks(nb);
                            for (uint64_t bi = 0; bi < nb; ++bi)
                                blocks[bi] = PqBlock{0, (uint32_t)(bi * PQ_BLOCK_ROWS), (uint32_t)std::min<uint64_t>(PQ_BLOCK_ROWS, n_out - bi * PQ_BLOCK_ROWS), 0u, 0u, 0u, 0u};
                            e.h2d(w.pq_blocks, blocks.data(), nb * sizeof(PqBlock));
                            Utf8Entries x;
                            x.stage = chunk;
                            x.blocks = w.pq_blocks;
                            x.n_blocks = (int64_t)nb;
                            x.row_ent = w.row_ent + (uint64_t)u * w.bound;
                            x.block_bytes = w.block_bytes + (uint64_t)u * (w.blocks + 1);
                            x.block_base = w.block_base + (uint64_t)u * (w.blocks + 1);
                            ++u;
                            append_utf8_from_entries(e, c, x, (int64_t)n_out);  // sets n_rows
                            continue;
                        }
                        if (cols[j].kind == CSV_BOOL) {
                            append_bits_device(e, c.values, c.tail_vbyte, have, w.bwords + j * w.words, (int64_t)n_out, ci[j].btail);
                            c.value_bytes = (have + (int64_t)n_out + 7) / 8;
                        } else {
                            c.value_bytes = (have + (int64_t)n_out) * c.elem_bytes();
                        }
                        c.n_rows = have + (int64_t)n_out;
                    }
                    rows += (int64_t)n_out;
                }
                if (info.n_rec > 0) header = false;
                if (!is_last) {
                    carry = len - info.consumed;
                    carry_src = chunk + info.consumed;
                }
            }
        }
        if (rows_out) *rows_out = rows;
    } catch (...) {
        release_staging();
        throw;
    }
    release_staging();
    txn.commit();
}

}  // namespace tg
