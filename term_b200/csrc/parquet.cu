// Parquet column chunk -> HBM (SURVEY §8f.4): replaces the decode half of the reference's ParquetSource
// (sources/parquet.rs:150-230, DataFusion's ParquetExec) plus the Arrow host->device copy for one column.
//
// Split of work. The host walks the chunk's pages (Thrift compact PageHeaders), expands the definition levels
// (RLE / bit-packed hybrid at bit width 1: one bit per row = n/8 bytes, cheap) into the column's validity bitmap
// while the value bytes are already on their way to the device, and describes the value sections as blocks of up to
// 1024 rows. The device does the part that is proportional to the data: PLAIN stores only the non-NULL values, densely,
// so pq_expand_kernel scatters them to their row positions (Arrow layout) — one warp per block, rank of a row among
// the block's non-NULL rows from a ballot. Pages without NULLs are copied straight into place (no kernel).
//
// Dictionary-encoded chunks (what writers produce by default): the dictionary page's PLAIN values and the data pages'
// index streams (RLE / bit-packed hybrid) travel as they are; the host only walks the RUN HEADERS of the index streams (one
// varint per run, not per value) into a run table, and pq_expand_kernel looks every row's index up on the device — binary
// search of its run, bit extraction, dictionary gather — in the same pass that scatters the values to their rows.
// Snappy-compressed pages are decompressed on the host into the staging source (the raw format's tag stream is serial
// by construction); the levels of V2 pages are never compressed.
//
// BOOLEAN chunks become the bit-packed Arrow Boolean values: PLAIN sections (bit-packed, LSB first) and RLE sections
// (4-byte length, then an RLE / bit-packed hybrid stream at bit width 1) are staged as they are; pq_expand_bool_kernel
// writes 32 rows per ballot into the column's value bitmap. INT96 chunks (12-byte legacy Impala / Hive timestamps) become
// Int64 nanoseconds since the epoch, converted by pq_expand_kernel as it loads each value.
//
// Supported (everything else is TG_ERR_UNSUPPORTED, there is no host decode path): physical INT64 / DOUBLE /
// INT32 / FLOAT / INT96 / BOOLEAN and BYTE_ARRAY strings (below), codecs UNCOMPRESSED and SNAPPY, data pages V1 and V2, PLAIN / PLAIN_DICTIONARY / RLE_DICTIONARY values
// (a chunk may mix them: writers fall back to PLAIN when the dictionary grows too large; BOOLEAN: PLAIN and RLE), RLE definition levels, flat
// columns (max definition level 0 or 1, no repetition levels).
#include <dlfcn.h>

#include <algorithm>
#include <memory>
#include <mutex>
#include <cstring>
#include <exception>
#include <thread>

#include "engine.hpp"
#include "str_entries.cuh"

namespace tg {

// ------------------------------------------------------------------ Thrift compact protocol (read-only) ----
namespace {

struct Thrift {
    const uint8_t* p;
    const uint8_t* end;
    void need(size_t n) const {
        if ((size_t)(end - p) < n) throw Error(TG_ERR_INVALID_ARG, "Parquet page header is truncated");
    }
    uint8_t byte() {
        need(1);
        return *p++;
    }
    uint64_t varint() {
        uint64_t v = 0;
        for (int shift = 0; shift < 64; shift += 7) {
            const uint8_t b = byte();
            v |= (uint64_t)(b & 0x7f) << shift;
            if (!(b & 0x80)) return v;
        }
        throw Error(TG_ERR_INVALID_ARG, "Parquet page header: varint too long");
    }
    int64_t zigzag() {
        const uint64_t v = varint();
        return (int64_t)(v >> 1) ^ -(int64_t)(v & 1);
    }
    // returns false at STOP; type = compact wire type, id = field id
    bool field(int& type, int& id, int& last_id) {
        const uint8_t h = byte();
        if (h == 0) return false;
        type = h & 0x0f;
        const int delta = h >> 4;
        id = delta ? last_id + delta : (int)zigzag();
        last_id = id;
        return true;
    }
    void skip(int type, int depth = 0) {
        if (depth > 16) throw Error(TG_ERR_INVALID_ARG, "Parquet page header: nesting too deep");
        switch (type) {
            case 1: case 2: break;  // bool carried by the type nibble
            case 3: byte(); break;
            case 4: case 5: case 6: varint(); break;
            case 7: need(8); p += 8; break;
            case 8: {
                const uint64_t n = varint();
                need(n);
                p += n;
            } break;
            case 9: case 10: {
                const uint8_t h = byte();
                uint64_t n = h >> 4;
                const int et = h & 0x0f;
                if (n == 15) n = varint();
                for (uint64_t i = 0; i < n; ++i) {
                    if (et == 1 || et == 2) byte();  // list elements spell booleans out
                    else skip(et, depth + 1);
                }
            } break;
            case 11: {
                const uint64_t n = varint();
                if (n) {
                    const uint8_t kv = byte();
                    for (uint64_t i = 0; i < n; ++i) {
                        skip(kv >> 4, depth + 1);
                        skip(kv & 0x0f, depth + 1);
                    }
                }
            } break;
            case 12: {
                int t, id, last = 0;
                while (field(t, id, last)) skip(t, depth + 1);
            } break;
            default: throw Error(TG_ERR_INVALID_ARG, "Parquet page header: unknown Thrift type");
        }
    }
};

enum { PQ_DATA_PAGE = 0, PQ_INDEX_PAGE = 1, PQ_DICTIONARY_PAGE = 2, PQ_DATA_PAGE_V2 = 3 };
enum { PQ_ENC_PLAIN = 0, PQ_ENC_PLAIN_DICTIONARY = 2, PQ_ENC_RLE = 3, PQ_ENC_DELTA_BINARY_PACKED = 5, PQ_ENC_DELTA_LENGTH_BYTE_ARRAY = 6,
       PQ_ENC_DELTA_BYTE_ARRAY = 7, PQ_ENC_RLE_DICTIONARY = 8, PQ_ENC_BYTE_STREAM_SPLIT = 9 };
enum { PQ_CODEC_UNCOMPRESSED = 0, PQ_CODEC_SNAPPY = 1, PQ_CODEC_GZIP = 2, PQ_CODEC_BROTLI = 4, PQ_CODEC_ZSTD = 6, PQ_CODEC_LZ4_RAW = 7 };

std::string encoding_name(int32_t enc) {
    static const char* const names[] = {"PLAIN", "GROUP_VAR_INT", "PLAIN_DICTIONARY", "RLE", "BIT_PACKED", "DELTA_BINARY_PACKED",
                                        "DELTA_LENGTH_BYTE_ARRAY", "DELTA_BYTE_ARRAY", "RLE_DICTIONARY", "BYTE_STREAM_SPLIT"};
    const std::string num = std::to_string(enc);
    return enc >= 0 && enc < 10 ? std::string(names[enc]) + " (" + num + ")" : "encoding " + num;
}

// parquet.thrift: PageHeader {1 type, 2 uncompressed_page_size, 3 compressed_page_size, 4 crc, 5 data_page_header,
// 6 index_page_header, 7 dictionary_page_header, 8 data_page_header_v2}; DataPageHeader {1 num_values, 2 encoding,
// 3 definition_level_encoding, 4 repetition_level_encoding, 5 statistics}; DataPageHeaderV2 {1 num_values, 2 num_nulls,
// 3 num_rows, 4 encoding, 5 definition_levels_byte_length, 6 repetition_levels_byte_length, 7 is_compressed, 8 statistics}
size_t parse_page_header(const uint8_t* p, const uint8_t* end, tg_parquet_page& pg) {
    Thrift t{p, end};
    pg = tg_parquet_page{};
    pg.page_type = -1;
    pg.encoding = -1;
    pg.definition_level_encoding = -1;
    int type, id, last = 0;
    while (t.field(type, id, last)) {
        if (id == 1 && type == 5) pg.page_type = (int32_t)t.zigzag();
        else if (id == 2 && type == 5) pg.uncompressed_bytes = (int32_t)t.zigzag();
        else if (id == 3 && type == 5) pg.body_bytes = (int32_t)t.zigzag();
        else if ((id == 5 || id == 8) && type == 12) {
            const bool v2 = id == 8;
            pg.version = v2 ? 2 : 1;
            int ft, fid, flast = 0;
            while (t.field(ft, fid, flast)) {
                if (fid == 1 && ft == 5) pg.num_values = (int32_t)t.zigzag();
                else if (!v2 && fid == 2 && ft == 5) pg.encoding = (int32_t)t.zigzag();
                else if (!v2 && fid == 3 && ft == 5) pg.definition_level_encoding = (int32_t)t.zigzag();
                else if (v2 && fid == 2 && ft == 5) pg.num_nulls = (int32_t)t.zigzag();
                else if (v2 && fid == 4 && ft == 5) pg.encoding = (int32_t)t.zigzag();
                else if (v2 && fid == 5 && ft == 5) pg.definition_levels_bytes = (int32_t)t.zigzag();
                else if (v2 && fid == 6 && ft == 5) pg.repetition_levels_bytes = (int32_t)t.zigzag();
                else if (v2 && fid == 7 && (ft == 1 || ft == 2)) pg.is_compressed = ft == 1;
                else t.skip(ft);
            }
            if (v2) pg.definition_level_encoding = PQ_ENC_RLE;
        } else if (id == 7 && type == 12) {
            int ft, fid, flast = 0;
            while (t.field(ft, fid, flast)) {
                if (fid == 1 && ft == 5) pg.num_values = (int32_t)t.zigzag();
                else if (fid == 2 && ft == 5) pg.encoding = (int32_t)t.zigzag();
                else t.skip(ft);
            }
        } else {
            t.skip(type);
        }
    }
    if (pg.page_type < 0 || pg.body_bytes < 0) throw Error(TG_ERR_INVALID_ARG, "Parquet page header without type / size");
    return (size_t)(t.p - p);
}

// ---- bit helpers on a chunk-relative, LSB-first bitmap (callers keep 16 bytes of slack behind it). The level streams
// of sparse-NULL columns are millions of short runs, so both helpers work a 64-bit word at a time ----
inline void or_word(uint8_t* bits, int64_t pos, uint64_t v) {  // v's bits land at pos ..; (pos & 7) + width(v) <= 64
    uint64_t w;
    memcpy(&w, bits + (pos >> 3), 8);
    w |= v << (pos & 7);
    memcpy(bits + (pos >> 3), &w, 8);
}
void set_ones(uint8_t* bits, int64_t pos, int64_t count) {
    if (count >= 512) {  // long run: bytes in the middle
        while (pos & 7) {
            bits[pos >> 3] |= (uint8_t)(1u << (pos & 7));
            ++pos;
            --count;
        }
        const int64_t full = count / 8;
        memset(bits + (pos >> 3), 0xFF, (size_t)full);
        pos += full * 8;
        count -= full * 8;
    }
    while (count > 0) {
        const int take = (int)std::min<int64_t>(count, 56);
        or_word(bits, pos, (1ull << take) - 1ull);
        pos += take;
        count -= take;
    }
}
// copies nbits bits of src (from its bit 0) to bits[pos ..); src_end bounds the 8-byte loads
void put_bits(uint8_t* bits, int64_t pos, const uint8_t* src, int64_t nbits, const uint8_t* src_end) {
    while (nbits > 0) {
        const int take = (int)std::min<int64_t>(nbits, 56);
        uint64_t v = 0;
        if (src + 8 <= src_end) memcpy(&v, src, 8);
        else memcpy(&v, src, (size_t)std::min<int64_t>((take + 7) / 8, src_end - src));
        if (take < 64) v &= (1ull << take) - 1ull;
        or_word(bits, pos, v);
        pos += take;
        nbits -= take;
        src += 7;
    }
}
int64_t count_ones(const uint8_t* bits, int64_t lo, int64_t hi) {
    int64_t c = 0;
    while (lo < hi && (lo & 63)) {
        c += (bits[lo >> 3] >> (lo & 7)) & 1;
        ++lo;
    }
    for (; lo + 64 <= hi; lo += 64) {
        uint64_t w;
        memcpy(&w, bits + (lo >> 3), 8);
        c += __builtin_popcountll(w);
    }
    for (; lo < hi; ++lo) c += (bits[lo >> 3] >> (lo & 7)) & 1;
    return c;
}

// RLE / bit-packed hybrid, bit width 1 (Parquet "RLE" encoding of definition levels for a flat optional column):
// <varint header> then, header & 1 ? (header >> 1) groups of 8 values, one byte each : a run of (header >> 1) copies
// of the value in the next byte. Writes `n` levels as bits at bits[pos ..).
void decode_levels(const uint8_t* p, const uint8_t* end, uint8_t* bits, int64_t pos, int64_t n) {
    Thrift t{p, end};
    int64_t done = 0;
    while (done < n) {
        const uint64_t h = t.varint();
        if (h & 1) {
            const int64_t groups = (int64_t)(h >> 1);
            t.need((size_t)groups);
            const int64_t take = std::min<int64_t>(groups * 8, n - done);  // the last group may be padded
            put_bits(bits, pos + done, t.p, take, t.end);
            t.p += groups;
            done += take;
        } else {
            const int64_t run = (int64_t)(h >> 1);
            const uint8_t v = t.byte();
            if (v > 1) throw Error(TG_ERR_UNSUPPORTED, "Parquet: definition level > 1 (nested column)");
            const int64_t take = std::min<int64_t>(run, n - done);
            if (run == 0) throw Error(TG_ERR_INVALID_ARG, "Parquet: empty RLE run in the definition levels");
            if (v) set_ones(bits, pos + done, take);
            done += take;
        }
    }
}

// Snappy raw format (format_description.txt): varint uncompressed length, then elements tagged by their low two bits:
// 00 literal (length - 1 in the upper six bits, 60..63: that many extra length bytes), 01 copy with an 11-bit offset and
// a 4..11 byte length, 10 copy with a 16-bit offset, 11 copy with a 32-bit offset (length - 1 in the upper six bits).
// Copies may overlap their own output (run-length expansion), so they move byte by byte when offset < length.
size_t snappy_uncompressed_length(const uint8_t* src, size_t n, size_t* header_bytes) {
    uint64_t v = 0;
    size_t i = 0;
    for (int shift = 0; shift < 35; shift += 7) {
        if (i >= n) throw Error(TG_ERR_INVALID_ARG, "Parquet: truncated Snappy stream");
        const uint8_t b = src[i++];
        v |= (uint64_t)(b & 0x7f) << shift;
        if (!(b & 0x80)) {
            *header_bytes = i;
            return (size_t)v;
        }
    }
    throw Error(TG_ERR_INVALID_ARG, "Parquet: bad Snappy length");
}
size_t snappy_decompress(const uint8_t* src, size_t n, uint8_t* dst, size_t cap) {
    size_t ip = 0;
    const size_t total = snappy_uncompressed_length(src, n, &ip);
    if (total > cap) throw Error(TG_ERR_INVALID_ARG, "Parquet: Snappy page larger than its header says");
    size_t op = 0;
    auto bad = []() { throw Error(TG_ERR_INVALID_ARG, "Parquet: corrupt Snappy stream"); };
    while (ip < n) {
        const uint8_t tag = src[ip++];
        size_t len, off = 0;
        if ((tag & 3) == 0) {
            len = (size_t)(tag >> 2) + 1;
            if (len > 60) {
                const size_t extra = len - 60;
                if (ip + extra > n) bad();
                len = 0;
                for (size_t k = 0; k < extra; ++k) len |= (size_t)src[ip + k] << (8 * k);
                len += 1;
                ip += extra;
            }
            if (ip + len > n || op + len > total) bad();
            memcpy(dst + op, src + ip, len);
            ip += len;
            op += len;
            continue;
        }
        if ((tag & 3) == 1) {
            if (ip + 1 > n) bad();
            len = (size_t)((tag >> 2) & 7) + 4;
            off = ((size_t)(tag >> 5) << 8) | src[ip];
            ip += 1;
        } else if ((tag & 3) == 2) {
            if (ip + 2 > n) bad();
            len = (size_t)(tag >> 2) + 1;
            off = (size_t)src[ip] | ((size_t)src[ip + 1] << 8);
            ip += 2;
        } else {
            if (ip + 4 > n) bad();
            len = (size_t)(tag >> 2) + 1;
            off = (size_t)src[ip] | ((size_t)src[ip + 1] << 8) | ((size_t)src[ip + 2] << 16) | ((size_t)src[ip + 3] << 24);
            ip += 4;
        }
        if (off == 0 || off > op || op + len > total) bad();
        if (off >= len) memcpy(dst + op, dst + op - off, len);
        else
            for (size_t k = 0; k < len; ++k) dst[op + k] = dst[op + k - off];
        op += len;
    }
    if (op != total) bad();
    return total;
}

// One run of a dictionary-index stream (RLE / bit-packed hybrid at the page's bit width)
struct PqRun {
    uint32_t start;   // dense index (among the section's non-NULL values) of the run's first value
    uint32_t count;
    uint64_t data;    // RLE: the repeated index; bit-packed: byte offset of the packed groups in the staging buffer
    uint32_t bw;      // bit width of the page (0..32)
    uint32_t packed;  // 1: bit-packed, 0: RLE
};
// Walks the run headers of an RLE / bit-packed hybrid stream at bit width `bw`: <varint header> (header & 1 ? bit-packed
// groups of 8 : RLE run) until `n_values` are covered. `stage_off` = where p[0] sits in the staging buffer.
void parse_hybrid_runs(const uint8_t* p, const uint8_t* end, uint32_t bw, int64_t n_values, uint64_t stage_off, std::vector<PqRun>& runs) {
    Thrift t{p, end};
    int64_t done = 0;
    while (done < n_values) {
        const uint64_t h = t.varint();
        if (h & 1) {
            const uint64_t groups = h >> 1;
            const uint64_t bytes = groups * bw;
            if (groups == 0 || groups > ((uint64_t)1 << 40)) throw Error(TG_ERR_INVALID_ARG, "Parquet: bad bit-packed run");
            t.need((size_t)bytes);
            const int64_t take = std::min<int64_t>((int64_t)groups * 8, n_values - done);
            runs.push_back(PqRun{(uint32_t)done, (uint32_t)take, stage_off + (uint64_t)(t.p - p), bw, 1u});
            t.p += bytes;
            done += take;
        } else {
            const uint64_t run = h >> 1;
            if (run == 0) throw Error(TG_ERR_INVALID_ARG, "Parquet: empty RLE run in the dictionary indices");
            const int vb = (int)(bw + 7) / 8;
            t.need((size_t)vb);
            uint64_t v = 0;
            for (int k = 0; k < vb; ++k) v |= (uint64_t)t.p[k] << (8 * k);
            t.p += vb;
            const int64_t take = std::min<int64_t>((int64_t)run, n_values - done);
            runs.push_back(PqRun{(uint32_t)done, (uint32_t)take, v, bw, 0u});
            done += take;
        }
    }
}
// A dictionary-index stream: p[0] = bit width, then the hybrid runs
void parse_index_runs(const uint8_t* p, const uint8_t* end, int64_t n_values, uint64_t stage_off, std::vector<PqRun>& runs) {
    if (n_values == 0) return;
    if (p >= end) throw Error(TG_ERR_INVALID_ARG, "Parquet: empty dictionary-index section");
    const uint32_t bw = p[0];
    if (bw > 32) throw Error(TG_ERR_INVALID_ARG, "Parquet: dictionary index bit width > 32");
    parse_hybrid_runs(p + 1, end, bw, n_values, stage_off + 1, runs);
}
// An RLE-encoded BOOLEAN value section: a 4-byte little-endian length, then the hybrid runs at bit width 1 (no width byte)
void parse_bool_runs(const uint8_t* p, int64_t n_bytes, int64_t n_values, uint64_t stage_off, std::vector<PqRun>& runs) {
    if (n_values == 0) return;
    if (n_bytes < 4) throw Error(TG_ERR_INVALID_ARG, "Parquet: RLE BOOLEAN section shorter than its 4-byte length");
    uint32_t len;
    memcpy(&len, p, 4);
    if ((int64_t)len > n_bytes - 4) throw Error(TG_ERR_INVALID_ARG, "Parquet: RLE BOOLEAN length runs past the page");
    const size_t first = runs.size();
    parse_hybrid_runs(p + 4, p + 4 + len, 1, n_values, stage_off + 4, runs);
    for (size_t k = first; k < runs.size(); ++k)
        if (!runs[k].packed && runs[k].data > 1) throw Error(TG_ERR_INVALID_ARG, "Parquet: RLE BOOLEAN run of a value other than 0 / 1");
}

// INT96 (Impala / Hive / Spark timestamps): int64 nanoseconds of the day, then the int32 Julian day; nanoseconds since the
// epoch in wrapping int64 arithmetic (instants outside 1677 .. 2262 wrap, as in arrow-rs)
__host__ __device__ inline uint64_t pq_int96_ns(uint64_t nanos, int32_t julian_day) {
    return ((uint64_t)(int64_t)julian_day - 2440588ull) * 86400000000000ull + nanos;
}
uint64_t pq_int96_ns_host(const uint8_t* p) {
    uint64_t nanos;
    int32_t day;
    memcpy(&nanos, p, 8);
    memcpy(&day, p + 8, 4);
    return pq_int96_ns(nanos, day);
}

// ---- GZIP / ZSTD / LZ4_RAW / BROTLI pages: inflated on the host by the system's own codec libraries, bound at run time the first
// time a chunk needs one (dlopen, like libnccl: libtermgpu.so keeps no link-time dependency); Snappy stays hand-written above.
struct PqCodecLibs {
    std::mutex mu;
    bool tried[8] = {};
    // zlib
    struct ZStream {  // z_stream of zlib 1.x on LP64
        const uint8_t* next_in; unsigned avail_in; unsigned long total_in;
        uint8_t* next_out; unsigned avail_out; unsigned long total_out;
        const char* msg; void* state; void* zalloc; void* zfree; void* opaque; int data_type; unsigned long adler; unsigned long reserved;
    };
    int (*inflateInit2_)(ZStream*, int, const char*, int) = nullptr;
    int (*inflate)(ZStream*, int) = nullptr;
    int (*inflateEnd)(ZStream*) = nullptr;
    size_t (*ZSTD_decompress)(void*, size_t, const void*, size_t) = nullptr;
    unsigned (*ZSTD_isError)(size_t) = nullptr;
    int (*LZ4_decompress_safe)(const char*, char*, int, int) = nullptr;
    int (*BrotliDecoderDecompress)(size_t, const uint8_t*, size_t*, uint8_t*) = nullptr;
    static void* open_first(std::initializer_list<const char*> names) {
        for (const char* n : names)
            if (void* h = dlopen(n, RTLD_NOW | RTLD_LOCAL)) return h;
        return nullptr;
    }
    void bind(int codec) {
        std::lock_guard<std::mutex> g(mu);
        if (tried[codec]) return;
        tried[codec] = true;
        if (codec == PQ_CODEC_GZIP) {
            if (void* h = open_first({"libz.so.1", "libz.so"})) {
                inflateInit2_ = (decltype(inflateInit2_))dlsym(h, "inflateInit2_");
                inflate = (decltype(inflate))dlsym(h, "inflate");
                inflateEnd = (decltype(inflateEnd))dlsym(h, "inflateEnd");
            }
        } else if (codec == PQ_CODEC_ZSTD) {
            if (void* h = open_first({"libzstd.so.1", "libzstd.so"})) {
                ZSTD_decompress = (decltype(ZSTD_decompress))dlsym(h, "ZSTD_decompress");
                ZSTD_isError = (decltype(ZSTD_isError))dlsym(h, "ZSTD_isError");
            }
        } else if (codec == PQ_CODEC_LZ4_RAW) {
            if (void* h = open_first({"liblz4.so.1", "liblz4.so"})) LZ4_decompress_safe = (decltype(LZ4_decompress_safe))dlsym(h, "LZ4_decompress_safe");
        } else if (codec == PQ_CODEC_BROTLI) {
            if (void* h = open_first({"libbrotlidec.so.1", "libbrotlidec.so"}))
                BrotliDecoderDecompress = (decltype(BrotliDecoderDecompress))dlsym(h, "BrotliDecoderDecompress");
        }
    }
};
PqCodecLibs g_codecs;

bool codec_supported(int32_t codec) {
    return codec == PQ_CODEC_UNCOMPRESSED || codec == PQ_CODEC_SNAPPY || codec == PQ_CODEC_GZIP || codec == PQ_CODEC_ZSTD ||
           codec == PQ_CODEC_LZ4_RAW || codec == PQ_CODEC_BROTLI;
}

// one page body -> dst[0, cap): returns the uncompressed size (which must not exceed what the page header announced)
size_t page_decompress(int32_t codec, const uint8_t* src, size_t n, uint8_t* dst, size_t cap) {
    if (codec == PQ_CODEC_SNAPPY) return snappy_decompress(src, n, dst, cap);
    g_codecs.bind(codec);
    if (n > 0x7fffffffull || cap > 0x7fffffffull) throw Error(TG_ERR_UNSUPPORTED, "Parquet: page of 2 GiB or more");
    switch (codec) {
        case PQ_CODEC_GZIP: {
            if (!g_codecs.inflateInit2_ || !g_codecs.inflate || !g_codecs.inflateEnd)
                throw Error(TG_ERR_UNSUPPORTED, "Parquet: GZIP pages need libz.so.1, which this host does not have");
            PqCodecLibs::ZStream z;
            memset(&z, 0, sizeof z);
            // window bits 15 + 32: zlib and gzip wrappers are both accepted (parquet-mr writes gzip members)
            if (g_codecs.inflateInit2_(&z, 15 + 32, "1.2.11", (int)sizeof z) != 0) throw Error(TG_ERR_INTERNAL, "Parquet: inflateInit2 failed");
            z.next_in = src;
            z.avail_in = (unsigned)n;
            z.next_out = dst;
            z.avail_out = (unsigned)cap;
            const int rc = g_codecs.inflate(&z, 4 /* Z_FINISH */);
            const size_t got = (size_t)z.total_out;
            g_codecs.inflateEnd(&z);
            if (rc != 1 /* Z_STREAM_END */) throw Error(TG_ERR_INVALID_ARG, "Parquet: corrupt GZIP page (or larger than its header says)");
            return got;
        }
        case PQ_CODEC_ZSTD: {
            if (!g_codecs.ZSTD_decompress || !g_codecs.ZSTD_isError)
                throw Error(TG_ERR_UNSUPPORTED, "Parquet: ZSTD pages need libzstd.so.1, which this host does not have");
            const size_t got = g_codecs.ZSTD_decompress(dst, cap, src, n);
            if (g_codecs.ZSTD_isError(got)) throw Error(TG_ERR_INVALID_ARG, "Parquet: corrupt ZSTD page (or larger than its header says)");
            return got;
        }
        case PQ_CODEC_LZ4_RAW: {
            if (!g_codecs.LZ4_decompress_safe) throw Error(TG_ERR_UNSUPPORTED, "Parquet: LZ4_RAW pages need liblz4.so.1, which this host does not have");
            const int got = g_codecs.LZ4_decompress_safe((const char*)src, (char*)dst, (int)n, (int)cap);
            if (got < 0) throw Error(TG_ERR_INVALID_ARG, "Parquet: corrupt LZ4 page (or larger than its header says)");
            return (size_t)got;
        }
        case PQ_CODEC_BROTLI: {
            if (!g_codecs.BrotliDecoderDecompress)
                throw Error(TG_ERR_UNSUPPORTED, "Parquet: BROTLI pages need libbrotlidec.so.1, which this host does not have");
            size_t got = cap;
            if (g_codecs.BrotliDecoderDecompress(n, src, &got, dst) != 1 /* BROTLI_DECODER_RESULT_SUCCESS */)
                throw Error(TG_ERR_INVALID_ARG, "Parquet: corrupt BROTLI page (or larger than its header says)");
            return got;
        }
    }
    throw Error(TG_ERR_UNSUPPORTED, "Parquet: codec " + std::to_string(codec));
}

}  // namespace

// The value of dense index d of a hybrid stream: the last of runs [lo, hi) with start <= d, then its RLE value or the d-th
// packed value (two 32-bit loads; the staging buffer keeps slack behind every section)
__device__ __forceinline__ uint64_t pq_run_value(const uint8_t* __restrict__ stage, const PqRun* __restrict__ runs, uint32_t lo, uint32_t hi,
                                                 uint32_t d) {
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(&runs[mid].start) <= d) lo = mid;
        else hi = mid;
    }
    const PqRun run = runs[lo];
    uint64_t idx = run.data;
    if (run.packed) {
        const uint64_t bit = (uint64_t)(d - run.start) * run.bw;
        const uint64_t byte = run.data + (bit >> 3);
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(stage + (byte & ~(uint64_t)3));
        const uint64_t w = (uint64_t)__ldg(wp) | ((uint64_t)__ldg(wp + 1) << 32);
        const uint32_t sh = (uint32_t)((byte & 3) * 8 + (bit & 7));
        idx = run.bw ? ((w >> sh) & (((uint64_t)1 << run.bw) - 1ull)) : 0ull;
    }
    return idx;
}

// How pq_expand_kernel reads value i of a PLAIN section or a dictionary: the stored type as it is ...
template <typename V>
struct PqLoadNative {
    static __device__ __forceinline__ V at(const uint8_t* __restrict__ base, uint64_t i) { return __ldg(reinterpret_cast<const V*>(base) + i); }
};
// ... or a 12-byte INT96 converted to Int64 nanoseconds. Sections and the dictionary start 16-byte aligned, so every value
// is 4-byte aligned: three 32-bit loads
struct PqLoadInt96 {
    static __device__ __forceinline__ uint64_t at(const uint8_t* __restrict__ base, uint64_t i) {
        const uint32_t* p = reinterpret_cast<const uint32_t*>(base + i * 12);
        return pq_int96_ns((uint64_t)__ldg(p) | ((uint64_t)__ldg(p + 1) << 32), (int32_t)__ldg(p + 2));
    }
};

// One warp per block. Row r of the block is non-NULL iff its bit is set (bits == nullptr: a required column, every row
// is); its value is the (number of set bits before r in the block)-th of the block's dense source values — read directly
// (PLAIN) or through the section's index stream and the chunk's dictionary. NULL rows are written as 0 so the column is
// deterministic. Indices past the dictionary (a corrupt file) read its last entry: memory-safe, never out of bounds.
template <typename V, typename Load = PqLoadNative<V>>
__global__ void __launch_bounds__(PQ_THREADS) pq_expand_kernel(const uint8_t* __restrict__ stage, const uint8_t* __restrict__ bits,
                                                              const PqBlock* __restrict__ blocks, int64_t n_blocks, V* __restrict__ dst,
                                                              const PqRun* __restrict__ runs, const uint8_t* __restrict__ dict, uint32_t dict_count) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (PQ_THREADS / 32);
    for (int64_t b = (int64_t)blockIdx.x * (PQ_THREADS / 32) + (threadIdx.x >> 5); b < n_blocks; b += warps) {
        const PqBlock blk = blocks[b];
        const uint8_t* src = stage + blk.src_off;
        uint32_t running = 0;
        for (uint32_t i = 0; i < blk.n_rows; i += 32) {
            const bool in = i + lane < blk.n_rows;
            const uint64_t r = (uint64_t)blk.first_row + i + lane;
            const bool valid = in && (!bits || ((__ldg(bits + (r >> 3)) >> (r & 7)) & 1));
            const unsigned mask = __ballot_sync(0xffffffffu, valid);
            const uint32_t rank = running + __popc(mask & ((1u << lane) - 1u));
            V v = 0;
            if (valid) {
                if (blk.run_hi == 0) {
                    v = Load::at(src, rank);
                } else {
                    uint64_t idx = pq_run_value(stage, runs, blk.run_lo, blk.run_hi, blk.first_dense + rank);
                    if (idx >= dict_count) idx = dict_count - 1;
                    v = Load::at(dict, idx);
                }
            }
            if (in) dst[r] = v;
            running += __popc(mask);
        }
    }
}

// BOOLEAN values, one warp per block as above. A valid row's value is bit (block src_off + rank) of the staged PLAIN
// section (src_off is a BIT offset here) or the value of its run in the section's RLE stream; NULL rows read 0. One
// ballot gives the bits of 32 consecutive rows, OR-ed into the column's value bitmap at bit dst_bit0 + row: pages and
// appends start at any row, so a word may straddle two blocks (the host zeroed the new bytes first; OR order does not matter).
__global__ void __launch_bounds__(PQ_THREADS) pq_expand_bool_kernel(const uint8_t* __restrict__ stage, const uint8_t* __restrict__ bits,
                                                                   const PqBlock* __restrict__ blocks, int64_t n_blocks, uint32_t* __restrict__ dst,
                                                                   uint64_t dst_bit0, const PqRun* __restrict__ runs) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (PQ_THREADS / 32);
    for (int64_t b = (int64_t)blockIdx.x * (PQ_THREADS / 32) + (threadIdx.x >> 5); b < n_blocks; b += warps) {
        const PqBlock blk = blocks[b];
        uint32_t running = 0;
        for (uint32_t i = 0; i < blk.n_rows; i += 32) {
            const bool in = i + lane < blk.n_rows;
            const uint64_t r = (uint64_t)blk.first_row + i + lane;
            const bool valid = in && (!bits || ((__ldg(bits + (r >> 3)) >> (r & 7)) & 1));
            const unsigned mask = __ballot_sync(0xffffffffu, valid);
            const uint32_t rank = running + __popc(mask & ((1u << lane) - 1u));
            uint32_t v = 0;
            if (valid) {
                if (blk.run_hi == 0) {
                    const uint64_t sb = blk.src_off + rank;
                    v = (__ldg(stage + (sb >> 3)) >> (sb & 7)) & 1u;
                } else {
                    v = (uint32_t)pq_run_value(stage, runs, blk.run_lo, blk.run_hi, blk.first_dense + rank) & 1u;
                }
            }
            const unsigned out = __ballot_sync(0xffffffffu, v != 0);
            if (lane == 0 && out) {
                const uint64_t pos = dst_bit0 + blk.first_row + i;
                const uint32_t sh = (uint32_t)(pos & 31);
                atomicOr(dst + (pos >> 5), out << sh);
                if (sh && (out >> (32 - sh))) atomicOr(dst + (pos >> 5) + 1, out >> (32 - sh));
            }
            running += __popc(mask);
        }
    }
}

static std::vector<tg_parquet_page> walk_pages(const uint8_t* chunk, int64_t n_bytes) {
    if (!chunk || n_bytes < 0) throw Error(TG_ERR_INVALID_ARG, "NULL chunk");
    std::vector<tg_parquet_page> out;
    int64_t off = 0;
    while (off < n_bytes) {
        tg_parquet_page pg;
        const size_t hl = parse_page_header(chunk + off, chunk + n_bytes, pg);
        pg.header_offset = off;
        pg.body_offset = off + (int64_t)hl;
        if (pg.body_offset + pg.body_bytes > n_bytes) throw Error(TG_ERR_INVALID_ARG, "Parquet page runs past the column chunk");
        // every count / length below comes from the file: nothing negative, no level section longer than its page
        if (pg.num_values < 0 || pg.num_nulls < 0 || pg.uncompressed_bytes < 0)
            throw Error(TG_ERR_INVALID_ARG, "Parquet page header: negative value count or size");
        if (pg.definition_levels_bytes < 0 || pg.repetition_levels_bytes < 0 ||
            (int64_t)pg.definition_levels_bytes + (int64_t)pg.repetition_levels_bytes > (int64_t)pg.body_bytes)
            throw Error(TG_ERR_INVALID_ARG, "Parquet page header: level sections do not fit the page");
        out.push_back(pg);
        off = pg.body_offset + pg.body_bytes;
    }
    return out;
}

int32_t parquet_inspect_chunk(const uint8_t* chunk, int64_t n_bytes, tg_parquet_page* pages, int32_t cap) {
    const std::vector<tg_parquet_page> v = walk_pages(chunk, n_bytes);
    for (size_t i = 0; pages && i < v.size() && (int32_t)i < cap; ++i) pages[i] = v[i];
    return (int32_t)v.size();
}

namespace {
// the number of non-NULL rows among the `n` definition levels of one page
int64_t count_levels_set(const uint8_t* p, const uint8_t* end, int64_t n) {
    if (n <= 0) return 0;
    std::vector<uint8_t> bits((size_t)(n + 7) / 8 + 8, 0);
    decode_levels(p, end, bits.data(), 0, n);
    return count_ones(bits.data(), 0, n);
}

// ---- DELTA_BINARY_PACKED / DELTA_LENGTH_BYTE_ARRAY / DELTA_BYTE_ARRAY / BYTE_STREAM_SPLIT pages (parquet-format Encodings.md):
// their value streams are serial prefix sums / byte transposes; the host rewrites them into the PLAIN layout of the page
// (fixed width: little-endian values; BYTE_ARRAY: 4-byte length + bytes) and the common PLAIN path takes it from there.
// Decodes one DELTA_BINARY_PACKED stream: <block size> <miniblocks per block> <total count> <first value (zigzag)>, then per
// block <min delta (zigzag)> <bit widths> <miniblocks>; values wrap in 64 bits (INT32 columns keep the low 32). Returns the
// end of the stream.
// `expect` >= 0: the count the page's levels announce — a stream that disagrees is refused before anything is allocated.
const uint8_t* delta_binary_unpack(const uint8_t* p, const uint8_t* end, std::vector<int64_t>& out, int64_t expect = -1) {
    Thrift t{p, end};
    const uint64_t block = t.varint(), minis = t.varint(), total = t.varint();
    uint64_t last = (uint64_t)t.zigzag();
    // (block sizes are 128 .. a few thousand in every writer; the bound keeps per_mini * bit width far from 64-bit overflow)
    if (block == 0 || block % 128 != 0 || block > ((uint64_t)1 << 24) || minis == 0 || block % minis != 0 || (block / minis) % 32 != 0 || minis > 512)
        throw Error(TG_ERR_INVALID_ARG, "Parquet: malformed DELTA_BINARY_PACKED header");
    if (expect >= 0 && total != (uint64_t)expect)
        throw Error(TG_ERR_INVALID_ARG, "Parquet: page holds " + std::to_string(total) + " encoded values, its levels say " + std::to_string(expect));
    if (total > (uint64_t)(end - p) * 64 + 1) throw Error(TG_ERR_INVALID_ARG, "Parquet: DELTA_BINARY_PACKED count does not fit the page");
    const uint64_t per_mini = block / minis;
    out.clear();
    out.reserve((size_t)total);
    if (total > 0) out.push_back((int64_t)last);
    while (out.size() < total) {
        const uint64_t min_delta = (uint64_t)t.zigzag();
        t.need((size_t)minis);
        const uint8_t* widths = t.p;
        t.p += minis;
        for (uint64_t m = 0; m < minis && out.size() < total; ++m) {
            const uint32_t bw = widths[m];
            if (bw > 64) throw Error(TG_ERR_INVALID_ARG, "Parquet: DELTA_BINARY_PACKED bit width above 64");
            const size_t bytes = (size_t)(per_mini * bw / 8);
            t.need(bytes);
            for (uint64_t i = 0; i < per_mini && out.size() < total; ++i) {
                uint64_t d = 0;
                if (bw) {
                    const uint64_t bit = i * bw;
                    const size_t byte = (size_t)(bit >> 3);
                    const uint32_t sh = (uint32_t)(bit & 7);
                    uint8_t buf[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
                    memcpy(buf, t.p + byte, std::min<size_t>(9, bytes - byte));
                    uint64_t lo;
                    memcpy(&lo, buf, 8);
                    d = lo >> sh;
                    if (sh && bw + sh > 64) d |= (uint64_t)buf[8] << (64 - sh);
                    if (bw < 64) d &= ((uint64_t)1 << bw) - 1;
                }
                last = last + min_delta + d;
                out.push_back((int64_t)last);
            }
            t.p += bytes;
        }
    }
    return t.p;
}

// one page's value section (n_present non-NULL values) of `encoding` -> PLAIN layout appended to `out`
void decode_to_plain(int32_t encoding, size_t elem_w, const uint8_t* p, int64_t n_bytes, int64_t n_present, std::vector<uint8_t>& out) {
    const uint8_t* end = p + n_bytes;
    std::vector<int64_t> a, b;
    auto need_count = [&](size_t got) {
        if ((int64_t)got != n_present) throw Error(TG_ERR_INVALID_ARG, "Parquet: page holds " + std::to_string(got) + " encoded values, its levels say " + std::to_string(n_present));
    };
    switch (encoding) {
        case PQ_ENC_DELTA_BINARY_PACKED: {
            if (elem_w != 4 && elem_w != 8) throw Error(TG_ERR_UNSUPPORTED, "Parquet: DELTA_BINARY_PACKED on a non-integer column");
            if (n_present == 0) return;
            delta_binary_unpack(p, end, a, n_present);
            need_count(a.size());
            const size_t at = out.size();
            out.resize(at + a.size() * elem_w);
            for (size_t i = 0; i < a.size(); ++i) memcpy(out.data() + at + i * elem_w, &a[i], elem_w);  // (little endian: the low bytes)
        } break;
        case PQ_ENC_BYTE_STREAM_SPLIT: {
            if (elem_w != 4 && elem_w != 8) throw Error(TG_ERR_UNSUPPORTED, "Parquet: BYTE_STREAM_SPLIT on a variable-width column");
            if (n_bytes != n_present * (int64_t)elem_w) throw Error(TG_ERR_INVALID_ARG, "Parquet: BYTE_STREAM_SPLIT page size does not match its value count");
            const size_t at = out.size();
            out.resize(at + (size_t)n_bytes);
            for (size_t k = 0; k < elem_w; ++k)
                for (int64_t i = 0; i < n_present; ++i) out[at + (size_t)i * elem_w + k] = p[k * (size_t)n_present + (size_t)i];
        } break;
        case PQ_ENC_DELTA_LENGTH_BYTE_ARRAY: {
            if (elem_w != 0) throw Error(TG_ERR_UNSUPPORTED, "Parquet: DELTA_LENGTH_BYTE_ARRAY on a fixed-width column");
            if (n_present == 0) return;
            const uint8_t* q = delta_binary_unpack(p, end, a, n_present);
            need_count(a.size());
            for (int64_t len : a) {
                if (len < 0 || len > end - q) throw Error(TG_ERR_INVALID_ARG, "Parquet: DELTA_LENGTH_BYTE_ARRAY value runs past the page");
                const uint32_t l32 = (uint32_t)len;
                out.insert(out.end(), (const uint8_t*)&l32, (const uint8_t*)&l32 + 4);
                out.insert(out.end(), q, q + len);
                q += len;
            }
        } break;
        case PQ_ENC_DELTA_BYTE_ARRAY: {
            if (elem_w != 0) throw Error(TG_ERR_UNSUPPORTED, "Parquet: DELTA_BYTE_ARRAY on a fixed-width column");
            if (n_present == 0) return;
            const uint8_t* q = delta_binary_unpack(p, end, a, n_present);  // prefix lengths
            q = delta_binary_unpack(q, end, b, n_present);                 // suffix lengths, then the suffix bytes
            need_count(a.size());
            need_count(b.size());
            size_t prev_at = 0, prev_len = 0;  // the previous value inside `out` (after its length prefix)
            for (size_t i = 0; i < a.size(); ++i) {
                const int64_t pre = a[i], suf = b[i];
                if (pre < 0 || (size_t)pre > prev_len || suf < 0 || suf > end - q || pre + suf > 0x7fffffffll)
                    throw Error(TG_ERR_INVALID_ARG, "Parquet: DELTA_BYTE_ARRAY value runs past the page or its predecessor");
                const uint32_t l32 = (uint32_t)(pre + suf);
                const size_t at = out.size();
                out.resize(at + 4 + (size_t)l32);
                memcpy(out.data() + at, &l32, 4);
                if (pre) memmove(out.data() + at + 4, out.data() + prev_at, (size_t)pre);
                memcpy(out.data() + at + 4 + pre, q, (size_t)suf);
                q += suf;
                prev_at = at + 4;
                prev_len = l32;
            }
        } break;
        default: throw Error(TG_ERR_UNSUPPORTED, "Parquet: value encoding " + std::to_string(encoding));
    }
}
bool encoding_rewritten_on_host(int32_t enc) {
    return enc == PQ_ENC_DELTA_BINARY_PACKED || enc == PQ_ENC_DELTA_LENGTH_BYTE_ARRAY || enc == PQ_ENC_DELTA_BYTE_ARRAY || enc == PQ_ENC_BYTE_STREAM_SPLIT;
}

struct PqSection {
    int64_t first_row, n_rows;
    const uint8_t* values;
    int64_t values_bytes;
    const uint8_t* levels;
    int64_t levels_bytes;
    bool dict;
    bool rle;  // BOOLEAN values in the RLE encoding
};
struct PqChunk {
    std::vector<PqSection> secs;
    std::vector<uint8_t> inflated;       // the uncompressed bodies of Snappy pages (sections point into it)
    std::vector<std::unique_ptr<std::vector<uint8_t>>> rewritten;  // PLAIN rewrites of DELTA / BYTE_STREAM_SPLIT value sections
    const uint8_t* dict_values = nullptr;
    int64_t dict_bytes = 0, dict_count = 0;
    bool any_dict = false;
};
// Cuts a data page's uncompressed body into its definition levels and its values. V1: a 4-byte length and the levels (when
// `levels`: an optional column), then the values; V2: the level sections the header sizes, then the values.
void split_levels(const tg_parquet_page& pg, const uint8_t* body, int64_t body_bytes, bool levels, PqSection& s) {
    int64_t lev_at = 0, lev_len = 0;
    if (pg.version == 2) {
        if (pg.repetition_levels_bytes != 0) throw Error(TG_ERR_UNSUPPORTED, "Parquet: repeated column");
        lev_len = pg.definition_levels_bytes;
    } else if (levels) {
        if (body_bytes < 4) throw Error(TG_ERR_INVALID_ARG, "Parquet: data page too short");
        uint32_t len;
        memcpy(&len, body, 4);
        if ((int64_t)len > body_bytes - 4) throw Error(TG_ERR_INVALID_ARG, "Parquet: definition levels run past the page");
        lev_at = 4;
        lev_len = len;
    }
    s.levels = levels ? body + lev_at : nullptr;
    s.levels_bytes = levels ? lev_len : 0;
    s.values = body + lev_at + lev_len;
    s.values_bytes = body_bytes - lev_at - lev_len;
    if (s.values_bytes < 0) throw Error(TG_ERR_INVALID_ARG, "Parquet: definition levels run past the page");
}
// width in the file of one fixed-width value of a chunk handed over as `dtype` (0: BYTE_ARRAY, and BOOLEAN's bits)
size_t source_width(int32_t dtype) {
    return dtype == TG_PQ_INT96 ? 12 : (dtype == TG_INT64 || dtype == TG_FLOAT64) ? 8 : (dtype == TG_INT32 || dtype == TG_FLOAT32) ? 4 : 0;
}

// Every page body as UNCOMPRESSED bytes (a view of the chunk, or of `inflated` for Snappy pages), cut into its level and
// value sections. dtype: the chunk's type as tg_table_append_parquet_chunk received it.
void collect_sections(const uint8_t* chunk, int64_t n_bytes, int32_t codec, int32_t max_def_level, int64_t num_values, int32_t dtype, PqChunk& out) {
    const size_t elem_w = source_width(dtype);
    const std::vector<tg_parquet_page> pages = walk_pages(chunk, n_bytes);
    {
        size_t need = 0;
        for (auto& pg : pages)
            if (codec != PQ_CODEC_UNCOMPRESSED && pg.page_type != PQ_INDEX_PAGE) need += (size_t)pg.uncompressed_bytes + 16;
        out.inflated.resize(need);
    }
    size_t inflated_used = 0;
    int64_t rows = 0;
    for (auto& pg : pages) {
        if (pg.page_type == PQ_INDEX_PAGE) continue;
        if (pg.page_type != PQ_DATA_PAGE && pg.page_type != PQ_DATA_PAGE_V2 && pg.page_type != PQ_DICTIONARY_PAGE)
            throw Error(TG_ERR_UNSUPPORTED, "Parquet: unknown page type");
        // the uncompressed body: V1 and dictionary pages are compressed as a whole, V2 keeps its level sections plain
        const uint8_t* body = chunk + pg.body_offset;
        int64_t body_bytes = pg.body_bytes;
        const int64_t plain_head = pg.page_type == PQ_DATA_PAGE_V2 ? (int64_t)pg.definition_levels_bytes + pg.repetition_levels_bytes : 0;
        const bool compressed = codec != PQ_CODEC_UNCOMPRESSED && (pg.page_type != PQ_DATA_PAGE_V2 || pg.is_compressed);
        if (compressed) {
            if ((int64_t)pg.uncompressed_bytes < plain_head) throw Error(TG_ERR_INVALID_ARG, "Parquet: page sizes do not fit its level sections");
            uint8_t* o = out.inflated.data() + inflated_used;
            memcpy(o, body, (size_t)plain_head);
            const size_t got = pg.body_bytes > plain_head
                                   ? page_decompress(codec, body + plain_head, (size_t)(pg.body_bytes - plain_head), o + plain_head,
                                                     (size_t)(pg.uncompressed_bytes - plain_head))
                                   : 0;
            body = o;
            body_bytes = plain_head + (int64_t)got;
            inflated_used += (size_t)pg.uncompressed_bytes + 16;
        }
        if (pg.page_type == PQ_DICTIONARY_PAGE) {
            if (dtype == TG_BOOL) throw Error(TG_ERR_UNSUPPORTED, "Parquet: dictionary-encoded BOOLEAN chunk (PLAIN and RLE values only)");
            if (pg.encoding != PQ_ENC_PLAIN && pg.encoding != PQ_ENC_PLAIN_DICTIONARY)
                throw Error(TG_ERR_UNSUPPORTED, "Parquet: dictionary page encoding " + std::to_string(pg.encoding));
            if (out.dict_values) throw Error(TG_ERR_INVALID_ARG, "Parquet: more than one dictionary page in a column chunk");
            if (elem_w && (int64_t)pg.num_values * (int64_t)elem_w > body_bytes)
                throw Error(TG_ERR_INVALID_ARG, "Parquet: dictionary page shorter than its value count");
            out.dict_values = body;
            out.dict_bytes = body_bytes;
            out.dict_count = pg.num_values;
            continue;
        }
        const bool is_dict = pg.encoding == PQ_ENC_RLE_DICTIONARY || pg.encoding == PQ_ENC_PLAIN_DICTIONARY;
        const bool is_rle = dtype == TG_BOOL && pg.encoding == PQ_ENC_RLE;
        if (dtype == TG_BOOL && pg.encoding != PQ_ENC_PLAIN && !is_rle)
            throw Error(TG_ERR_UNSUPPORTED, "Parquet: BOOLEAN values encoded " + encoding_name(pg.encoding) + " (PLAIN and RLE only)");
        if (dtype == TG_PQ_INT96 && pg.encoding != PQ_ENC_PLAIN && !is_dict)
            throw Error(TG_ERR_UNSUPPORTED, "Parquet: INT96 values encoded " + encoding_name(pg.encoding) + " (PLAIN and dictionary only)");
        if (!is_dict && !is_rle && pg.encoding != PQ_ENC_PLAIN && !encoding_rewritten_on_host(pg.encoding))
            throw Error(TG_ERR_UNSUPPORTED, "Parquet: value encoding " + std::to_string(pg.encoding) +
                                                " (PLAIN, dictionary, DELTA_* and BYTE_STREAM_SPLIT encodings only)");
        if (max_def_level > 0 && pg.definition_level_encoding != PQ_ENC_RLE)
            throw Error(TG_ERR_UNSUPPORTED, "Parquet: definition levels not RLE-encoded");
        PqSection s{rows, pg.num_values, nullptr, 0, nullptr, 0, is_dict, is_rle};
        split_levels(pg, body, body_bytes, max_def_level > 0, s);
        if (encoding_rewritten_on_host(pg.encoding)) {
            // the number of values present = the page's rows minus its NULLs (counted from the levels when the header has no count)
            int64_t present = pg.num_values;
            if (max_def_level > 0) {
                if (pg.version == 2) present -= pg.num_nulls;
                else present = count_levels_set(s.levels, s.levels + s.levels_bytes, pg.num_values);
            }
            out.rewritten.push_back(std::make_unique<std::vector<uint8_t>>());
            decode_to_plain(pg.encoding, elem_w, s.values, s.values_bytes, present, *out.rewritten.back());
            s.values = out.rewritten.back()->data();
            s.values_bytes = (int64_t)out.rewritten.back()->size();
        }
        rows += pg.num_values;
        out.any_dict = out.any_dict || is_dict;
        out.secs.push_back(s);
    }
    if (rows != num_values) throw Error(TG_ERR_INVALID_ARG, "Parquet: pages hold " + std::to_string(rows) + " values, the chunk metadata says " + std::to_string(num_values));
    if (!out.dict_values) out.dict_count = 0;  // (a dictionary-encoded page needs one unless all its rows are NULL: checked with the levels)
}

// entries: pq_str_ent / PQ_STR_MAX_LEN (str_entries.cuh)
// walks `count` PLAIN BYTE_ARRAY values at p (length prefixes interleaved) into entries; stage_off = where p sits in staging
void walk_plain_strings(const uint8_t* p, int64_t n_bytes, int64_t count, uint64_t stage_off, std::vector<uint64_t>& ents) {
    int64_t pos = 0;
    for (int64_t i = 0; i < count; ++i) {
        if (pos + 4 > n_bytes) throw Error(TG_ERR_INVALID_ARG, "Parquet: BYTE_ARRAY page is truncated");
        uint32_t len;
        memcpy(&len, p + pos, 4);
        pos += 4;
        if ((int64_t)len > n_bytes - pos) throw Error(TG_ERR_INVALID_ARG, "Parquet: BYTE_ARRAY value runs past its page");
        if (len > PQ_STR_MAX_LEN) throw Error(TG_ERR_UNSUPPORTED, "Parquet: string value of 16 MiB or more");
        ents.push_back(pq_str_ent(stage_off + (uint64_t)pos, len));
        pos += len;
    }
}

// What a chunk's values are; decides a block's src_off and what a section without dictionary indices gets
enum PqKind { PQ_KIND_FIXED, PQ_KIND_BOOL, PQ_KIND_STR };

// A chunk's sections staged on the device and described for the expand / locate kernels
struct PqStaged {
    uint8_t* stage = nullptr;       // every section's value bytes, then the dictionary; freed through deferred_free
    std::vector<int64_t> sec_off;   // each section's offset in `stage`
    size_t dict_off = 0;
    std::vector<uint8_t> bits;      // chunk-relative validity (16 bytes of slack); empty: a required column
    std::vector<PqBlock> blocks;
    std::vector<PqRun> runs;        // dictionary-index and RLE BOOLEAN streams
    std::vector<std::pair<uint32_t, uint32_t>> sec_runs;  // each section's runs [lo, hi) in `runs`
    std::vector<uint64_t> plain_ents;  // BYTE_ARRAY: one entry per value of the PLAIN sections
};

// Section i: its levels -> st.bits, its blocks of <= PQ_BLOCK_ROWS rows (non-NULL counts from popcounts of the bits), and
// the run table of its dictionary indices / RLE BOOLEAN values, or the check / entries of its PLAIN values
void cut_section(const PqChunk& pc, size_t i, PqKind kind, size_t sw, PqStaged& st) {
    const PqSection& s = pc.secs[i];
    const bool levels = !st.bits.empty();
    const uint64_t off = (uint64_t)st.sec_off[i];
    if (levels) decode_levels(s.levels, s.levels + s.levels_bytes, st.bits.data(), s.first_row, s.n_rows);
    const uint32_t run_lo = (uint32_t)st.runs.size();
    const size_t blk_lo = st.blocks.size();
    const uint64_t ent_lo = (uint64_t)st.plain_ents.size();
    int64_t prefix = 0;
    for (int64_t r = 0; r < s.n_rows; r += PQ_BLOCK_ROWS) {
        const int64_t nr = std::min<int64_t>(PQ_BLOCK_ROWS, s.n_rows - r);
        // the block's first value: an index into plain_ents (BYTE_ARRAY), a bit offset (BOOLEAN) or a byte offset in `stage`
        const uint64_t src = kind == PQ_KIND_STR ? ent_lo + (uint64_t)prefix
                             : kind == PQ_KIND_BOOL ? off * 8 + (uint64_t)prefix
                                                    : off + (uint64_t)prefix * sw;
        st.blocks.push_back(PqBlock{src, (uint32_t)(s.first_row + r), (uint32_t)nr, (uint32_t)prefix, 0u, 0u, 0u});
        prefix += levels ? count_ones(st.bits.data(), s.first_row + r, s.first_row + r + nr) : nr;
    }
    if (s.dict) {
        if (prefix > 0 && pc.dict_count <= 0) throw Error(TG_ERR_INVALID_ARG, "Parquet: dictionary-encoded page without a dictionary page");
        parse_index_runs(s.values, s.values + s.values_bytes, prefix, off, st.runs);
    } else if (s.rle) {
        parse_bool_runs(s.values, s.values_bytes, prefix, off, st.runs);
    } else if (kind == PQ_KIND_STR) {
        walk_plain_strings(s.values, s.values_bytes, prefix, off, st.plain_ents);
    } else if (kind == PQ_KIND_BOOL ? s.values_bytes < (prefix + 7) / 8 : prefix * (int64_t)sw != s.values_bytes) {
        throw Error(TG_ERR_INVALID_ARG, "Parquet: PLAIN page holds " + std::to_string(s.values_bytes) + " value bytes for " +
                                            std::to_string(prefix) + " non-null rows");
    }
    const uint32_t run_hi = (uint32_t)st.runs.size();
    st.sec_runs[i] = {run_lo, run_hi};
    if (s.dict || s.rle)
        for (size_t k = blk_lo; k < st.blocks.size(); ++k) {
            st.blocks[k].run_lo = run_lo;
            st.blocks[k].run_hi = run_hi > run_lo ? run_hi : run_lo + 1;  // (an all-NULL section has no runs: never looked up)
        }
}

// Stages a chunk: every section's value bytes at a 16-byte aligned place of one device block, then the dictionary
// (dict_count * sw bytes of fixed-width values, or the whole page body of a BYTE_ARRAY dictionary), then 64 bytes of
// slack. Staging a pageable source is a host memcpy into the pinned ring per piece, so a helper thread cuts the sections
// (cut_section) meanwhile. sw: the file width of a fixed-width value.
PqStaged stage_chunk(Engine& e, const PqChunk& pc, PqKind kind, size_t sw, int32_t max_def_level, int64_t num_values) {
    PqStaged st;
    size_t stage_bytes = 0;
    for (const PqSection& s : pc.secs) {
        st.sec_off.push_back((int64_t)stage_bytes);
        stage_bytes += r16((size_t)s.values_bytes);
    }
    st.dict_off = stage_bytes;
    const size_t dict_b = kind == PQ_KIND_STR ? (size_t)pc.dict_bytes : (size_t)pc.dict_count * sw;
    stage_bytes += r16(dict_b) + 64;
    if (stage_bytes >= PQ_STAGE_MAX) throw Error(TG_ERR_UNSUPPORTED, "Parquet: column chunk of 1 TiB or more");
    st.sec_runs.resize(pc.secs.size());
    std::exception_ptr cut_err;
    std::thread helper([&]() {
        try {
            if (max_def_level > 0) st.bits.assign((size_t)(num_values + 7) / 8 + 16, 0);
            st.blocks.reserve((size_t)num_values / PQ_BLOCK_ROWS + pc.secs.size() + 1);
            for (size_t i = 0; i < pc.secs.size(); ++i) cut_section(pc, i, kind, sw, st);
        } catch (...) {
            cut_err = std::current_exception();
        }
    });
    struct Join {
        std::thread& t;
        ~Join() {
            if (t.joinable()) t.join();
        }
    } join{helper};
    st.stage = e.dev_alloc(stage_bytes);
    e.deferred_free.emplace_back(st.stage, stage_bytes);  // released by the next sync_copies(), also on the error paths
    for (size_t i = 0; i < pc.secs.size(); ++i)
        if (pc.secs[i].values_bytes) e.h2d(st.stage + st.sec_off[i], pc.secs[i].values, (size_t)pc.secs[i].values_bytes);
    if (dict_b) e.h2d(st.stage + st.dict_off, pc.dict_values, dict_b);
    helper.join();
    if (cut_err) std::rethrow_exception(cut_err);
    return st;
}

// Host mirror of pq_run_value: the value of dense index d of section i, from its runs and its host bytes
uint64_t pq_run_value_host(const PqChunk& pc, const PqStaged& st, size_t i, uint32_t d) {
    uint32_t lo = st.sec_runs[i].first, hi = st.sec_runs[i].second;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (st.runs[mid].start <= d) lo = mid;
        else hi = mid;
    }
    const PqRun& run = st.runs[lo];
    if (!run.packed) return run.data;
    const PqSection& s = pc.secs[i];
    const uint64_t bit = (uint64_t)(d - run.start) * run.bw;
    const size_t byte = (size_t)(run.data - (uint64_t)st.sec_off[i] + (bit >> 3));
    uint64_t w = 0;
    memcpy(&w, s.values + byte, std::min<size_t>(8, (size_t)s.values_bytes - byte));
    return run.bw ? (w >> (bit & 7)) & (((uint64_t)1 << run.bw) - 1ull) : 0ull;
}

// The column's first values (at most 4096; INT96 converted, so the pivot is the one of the same instants delivered as
// timestamp[ns]), which the pivot of the shifted sums is chosen from like on the Arrow path (same K, bit-identical sums):
// the first section with values, its PLAIN values or the dictionary entries its indices name
std::vector<uint64_t> head_values(const PqChunk& pc, const PqStaged& st, size_t sw, bool int96) {
    auto at = [&](const uint8_t* p) {
        uint64_t v;
        if (int96) v = pq_int96_ns_host(p);
        else memcpy(&v, p, 8);
        return v;
    };
    std::vector<uint64_t> head;
    for (size_t i = 0; i < pc.secs.size() && head.empty(); ++i) {
        const PqSection& s = pc.secs[i];
        if (!s.dict) {
            const int64_t n = std::min<int64_t>(s.values_bytes / (int64_t)sw, 4096);
            for (int64_t k = 0; k < n; ++k) head.push_back(at(s.values + (size_t)k * sw));
        } else if (st.sec_runs[i].second > st.sec_runs[i].first) {
            const PqRun& last = st.runs[st.sec_runs[i].second - 1];
            const uint32_t n = std::min<uint32_t>(last.start + last.count, 4096);
            for (uint32_t d = 0; d < n; ++d) {
                const uint64_t idx = std::min<uint64_t>(pq_run_value_host(pc, st, i, d), (uint64_t)pc.dict_count - 1);
                head.push_back(at(pc.dict_values + (size_t)idx * sw));
            }
        }
    }
    return head;
}

// One device block of tables, on deferred_free from the start: bits | blocks | runs, then the caller's `extra` tables
// ({host bytes or nullptr for device scratch, size}), each 16-byte aligned, 64 bytes of slack. Returns where each starts
// (bits: nullptr for a required column).
std::vector<uint8_t*> upload_tables(Engine& e, const PqStaged& st, int64_t num_values,
                                    std::initializer_list<std::pair<const void*, size_t>> extra = {}) {
    std::vector<std::pair<const void*, size_t>> parts = {{st.bits.data(), st.bits.empty() ? 0 : (size_t)(num_values + 7) / 8},
                                                         {st.blocks.data(), st.blocks.size() * sizeof(PqBlock)},
                                                         {st.runs.data(), st.runs.size() * sizeof(PqRun)}};
    parts.insert(parts.end(), extra);
    size_t total = 64;
    for (auto& p : parts) total += r16(p.second);
    uint8_t* q = e.dev_alloc(total);
    e.deferred_free.emplace_back(q, total);
    std::vector<uint8_t*> at;
    for (auto& p : parts) {
        at.push_back(q);
        if (p.first && p.second) e.h2d(q, p.first, p.second);
        q += r16(p.second);
    }
    if (st.bits.empty()) at[0] = nullptr;
    return at;
}
}  // namespace

// Host-only: the validity bitmap (chunk-relative, LSB first, (num_values + 7) / 8 bytes) a flat optional column chunk
// decodes to, and its non-NULL count. The device path builds exactly this before it scatters the values.
int64_t parquet_chunk_validity(const uint8_t* chunk, int64_t n_bytes, int64_t num_values, uint8_t* out_bits) {
    const std::vector<tg_parquet_page> pages = walk_pages(chunk, n_bytes);
    std::vector<uint8_t> bits((size_t)(num_values + 7) / 8 + 16, 0);
    int64_t rows = 0;
    for (auto& pg : pages) {
        if (pg.page_type != PQ_DATA_PAGE && pg.page_type != PQ_DATA_PAGE_V2) continue;
        if (rows + pg.num_values > num_values) throw Error(TG_ERR_INVALID_ARG, "Parquet: more values than the chunk metadata says");
        PqSection s{};
        split_levels(pg, chunk + pg.body_offset, pg.body_bytes, true, s);
        decode_levels(s.levels, s.levels + s.levels_bytes, bits.data(), rows, pg.num_values);
        rows += pg.num_values;
    }
    if (out_bits) memcpy(out_bits, bits.data(), (size_t)(num_values + 7) / 8);
    return count_ones(bits.data(), 0, rows);
}

static void append_parquet_utf8(AppendTxn& txn, const std::string& name, int32_t max_def_level, int32_t codec, const uint8_t* chunk, int64_t n_bytes,
                                int64_t num_values);
static void append_parquet_fixed(AppendTxn& txn, const std::string& name, int32_t dtype, int32_t max_def_level, int32_t codec, const uint8_t* chunk,
                                 int64_t n_bytes, int64_t num_values);

void table_append_parquet_chunk(Table& t, const std::string& name, int32_t dtype, int32_t max_def_level, int32_t codec,
                                const uint8_t* chunk, int64_t n_bytes, int64_t num_values) {
    AppendTxn txn(t);
    if (!chunk || n_bytes <= 0 || num_values < 0) throw Error(TG_ERR_INVALID_ARG, "empty Parquet column chunk");
    if (!codec_supported(codec))
        throw Error(TG_ERR_UNSUPPORTED, "Parquet: codec " + std::to_string(codec) + " (UNCOMPRESSED, SNAPPY, GZIP, BROTLI, ZSTD and LZ4_RAW chunks are decoded)");
    if (max_def_level < 0 || max_def_level > 1) throw Error(TG_ERR_UNSUPPORTED, "Parquet: nested columns (max definition level > 1)");
    if (num_values >= ((int64_t)1 << 31)) throw Error(TG_ERR_UNSUPPORTED, "Parquet: column chunk with 2^31 or more values");
    if (dtype == TG_UTF8) append_parquet_utf8(txn, name, max_def_level, codec, chunk, n_bytes, num_values);
    else append_parquet_fixed(txn, name, dtype, max_def_level, codec, chunk, n_bytes, num_values);
    txn.commit();
}

// INT64 / DOUBLE / INT32 / FLOAT / INT96 / BOOLEAN chunks
static void append_parquet_fixed(AppendTxn& txn, const std::string& name, int32_t dtype, int32_t max_def_level, int32_t codec, const uint8_t* chunk,
                                 int64_t n_bytes, int64_t num_values) {
    Engine& e = txn.e;
    const bool is_bool = dtype == TG_BOOL, int96 = dtype == TG_PQ_INT96;
    if (dtype != TG_INT64 && dtype != TG_FLOAT64 && dtype != TG_INT32 && dtype != TG_FLOAT32 && !is_bool && !int96)
        throw Error(TG_ERR_UNSUPPORTED, "Parquet: only INT64 / DOUBLE / INT32 / FLOAT / INT96 / BOOLEAN / BYTE_ARRAY (Utf8) columns are decoded on the device");
    const int32_t stored = int96 ? TG_INT64 : dtype;
    if (int96) {  // an INT96 column is Timestamp(Nanosecond, None) and nothing else
        const Column* have_c = txn.t.find(name);
        if (have_c && !(have_c->src_type && strcmp(have_c->src_type, "Timestamp") == 0 && have_c->temporal_unit == 'n'))
            throw Error(TG_ERR_TYPE_MISMATCH, "column '" + name + "' was registered with a different type than INT96 (Timestamp(Nanosecond, None))");
    }
    Column& c = txn.column(name, stored);
    if (int96) {  // what tg_table_set_column_arrow_type(.., "tsn:") declares
        c.src_type = "Timestamp";
        c.src_unsigned = false;
        c.temporal = true;
        c.temporal_unit = 'n';
    }
    const int64_t have = c.n_rows;
    const size_t w = (size_t)c.elem_bytes(), sw = source_width(dtype);  // stored / file width of a value (Boolean: bits, 0)

    PqChunk pc;
    collect_sections(chunk, n_bytes, codec, max_def_level, num_values, dtype, pc);
    if (num_values == 0) return;

    // PLAIN pages of required columns go straight into place; everything else is staged and expanded by a kernel
    if (is_bool) e.dev_reserve(c.values, (size_t)(have + num_values + 7) / 8, (size_t)(have + 7) / 8);
    else e.dev_reserve(c.values, (size_t)(have + num_values) * w, (size_t)have * w);
    uint8_t* dst = c.values.p + (size_t)have * w;
    const bool direct = max_def_level == 0 && !pc.any_dict && sw == w && !is_bool;
    PqStaged st;
    if (direct) {
        for (auto& s : pc.secs) {
            if (s.values_bytes != s.n_rows * (int64_t)w) throw Error(TG_ERR_INVALID_ARG, "Parquet: PLAIN page size does not match its value count");
            e.h2d(dst + (size_t)s.first_row * w, s.values, (size_t)s.values_bytes);
        }
    } else {
        st = stage_chunk(e, pc, is_bool ? PQ_KIND_BOOL : PQ_KIND_FIXED, sw, max_def_level, num_values);
    }
    if (!c.pivot_set && (stored == TG_INT64 || stored == TG_FLOAT64)) {
        const std::vector<uint64_t> head = head_values(pc, st, sw, int96);
        if (!head.empty()) set_pivot_host(c, stored, (int64_t)head.size(), head.data(), nullptr, 0);
    }
    // validity through the common path (keeps the host mirror of a partial tail byte)
    append_validity(e, c, have, st.bits.empty() ? nullptr : st.bits.data(), 0, num_values);

    if (!direct) {
        // h2d of pageable memory returns once the bytes sit in the pinned ring, so `st` / `pc` may go out of scope
        const std::vector<uint8_t*> d = upload_tables(e, st, num_values);
        const int64_t nb = (int64_t)st.blocks.size();
        const int grid = pq_str_grid(e, nb);
        const PqBlock* d_blocks = reinterpret_cast<const PqBlock*>(d[1]);
        const PqRun* d_runs = reinterpret_cast<const PqRun*>(d[2]);
        const uint8_t* dict = st.stage + st.dict_off;
        if (is_bool) {
            // the kernel ORs whole words: the new bytes start at zero (the partial byte before them keeps its earlier rows)
            const size_t z0 = (size_t)(have + 7) / 8, z1 = (size_t)(have + num_values + 7) / 8;
            if (z1 > z0) TG_CUDA(cudaMemsetAsync(c.values.p + z0, 0, z1 - z0, e.copy_stream));
            pq_expand_bool_kernel<<<grid, PQ_THREADS, 0, e.copy_stream>>>(st.stage, d[0], d_blocks, nb, reinterpret_cast<uint32_t*>(c.values.p),
                                                                          (uint64_t)have, d_runs);
        } else if (int96) {
            pq_expand_kernel<uint64_t, PqLoadInt96><<<grid, PQ_THREADS, 0, e.copy_stream>>>(st.stage, d[0], d_blocks, nb, reinterpret_cast<uint64_t*>(dst),
                                                                                           d_runs, dict, (uint32_t)pc.dict_count);
        } else if (w == 8) {
            pq_expand_kernel<uint64_t><<<grid, PQ_THREADS, 0, e.copy_stream>>>(st.stage, d[0], d_blocks, nb, reinterpret_cast<uint64_t*>(dst), d_runs,
                                                                               dict, (uint32_t)pc.dict_count);
        } else {
            pq_expand_kernel<uint32_t><<<grid, PQ_THREADS, 0, e.copy_stream>>>(st.stage, d[0], d_blocks, nb, reinterpret_cast<uint32_t*>(dst), d_runs,
                                                                               dict, (uint32_t)pc.dict_count);
        }
        TG_CUDA(cudaGetLastError());
        e.launches += 1;
    }
    if (is_bool) {
        // host mirror of the value bitmap's last partial byte (table_append_host continues from it): its rows before this
        // chunk from the old mirror, the chunk's own (at most 7) rows decoded here from the host copies of the sections
        const int64_t total = have + num_values, lo = total & ~(int64_t)7;
        uint8_t tail = lo < have ? (uint8_t)(c.tail_vbyte & ((1u << (have - lo)) - 1u)) : 0;
        for (int64_t row = std::max(lo, have); row < total; ++row) {
            const int64_t r = row - have;
            if (!st.bits.empty() && !((st.bits[(size_t)(r >> 3)] >> (r & 7)) & 1)) continue;
            size_t i = pc.secs.size() - 1;
            while (pc.secs[i].first_row > r) --i;
            const PqSection& s = pc.secs[i];
            const int64_t d = st.bits.empty() ? r - s.first_row : count_ones(st.bits.data(), s.first_row, r);
            const uint64_t v = s.rle ? pq_run_value_host(pc, st, i, (uint32_t)d) : (uint64_t)(s.values[d >> 3] >> (d & 7));
            tail |= (uint8_t)((v & 1u) << (row - lo));
        }
        c.tail_vbyte = tail;
        c.value_bytes = (total + 7) / 8;
    } else {
        c.value_bytes = (have + num_values) * (int64_t)w;
    }
    c.n_rows = have + num_values;
}

// ---------------------------------------------------------------------------------------------------------------------
// BYTE_ARRAY (Utf8) chunks. A value is a 4-byte length followed by its bytes (PLAIN) or an index into a dictionary of such
// values; the Arrow layout wants int32 offsets (one more than rows) and the concatenated bytes. Three device steps:
//   pq_str_locate_kernel  per row: where its bytes sit in the staging buffer and how long they are — through the
//                         dictionary (index stream as for fixed-width columns) or the PLAIN section's entry table — and
//                         the byte total of every 1024-row block
//   pq_block_scan_kernel  exclusive scan of the block totals (one CTA)
//   pq_str_write_kernel   in-block scan of the lengths -> offsets, bytes copied to their place
// The host walks what is serial by construction: page headers, run headers, and the interleaved length prefixes of PLAIN
// pages (one entry {staging offset, length} per value); the dictionary page's own entries likewise (it is small).
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t pq_row_entry(const PqBlock& blk, uint32_t rank, const uint8_t* __restrict__ stage,
                                                 const PqRun* __restrict__ runs, const uint64_t* __restrict__ plain_ents,
                                                 const uint64_t* __restrict__ dict_ents, uint32_t dict_count) {
    if (blk.run_hi == 0) return __ldg(plain_ents + blk.src_off + rank);  // PLAIN: src_off = the block's first entry
    uint64_t idx = pq_run_value(stage, runs, blk.run_lo, blk.run_hi, blk.first_dense + rank);
    if (idx >= dict_count) idx = dict_count - 1;
    return __ldg(dict_ents + idx);
}

__global__ void __launch_bounds__(PQ_THREADS) pq_str_locate_kernel(const uint8_t* __restrict__ stage, const uint8_t* __restrict__ bits,
                                                                  const PqBlock* __restrict__ blocks, int64_t n_blocks,
                                                                  const PqRun* __restrict__ runs, const uint64_t* __restrict__ plain_ents,
                                                                  const uint64_t* __restrict__ dict_ents, uint32_t dict_count,
                                                                  uint64_t* __restrict__ row_ent, unsigned long long* __restrict__ block_bytes) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (PQ_THREADS / 32);
    for (int64_t b = (int64_t)blockIdx.x * (PQ_THREADS / 32) + (threadIdx.x >> 5); b < n_blocks; b += warps) {
        const PqBlock blk = blocks[b];
        uint32_t running = 0;
        unsigned long long total = 0;
        for (uint32_t i = 0; i < blk.n_rows; i += 32) {
            const bool in = i + lane < blk.n_rows;
            const uint64_t r = (uint64_t)blk.first_row + i + lane;
            const bool valid = in && (!bits || ((__ldg(bits + (r >> 3)) >> (r & 7)) & 1));
            const unsigned mask = __ballot_sync(0xffffffffu, valid);
            const uint32_t rank = running + __popc(mask & ((1u << lane) - 1u));
            uint64_t ent = 0;
            if (valid) ent = pq_row_entry(blk, rank, stage, runs, plain_ents, dict_ents, dict_count);
            if (in) row_ent[r] = ent;
            total += ent >> 40;
            running += __popc(mask);
        }
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) total += __shfl_xor_sync(0xffffffffu, total, m);
        if (lane == 0) block_bytes[b] = total;
    }
}

// one CTA: exclusive scan of the block totals; out[n] = the grand total
__global__ void __launch_bounds__(1024) pq_block_scan_kernel(const unsigned long long* __restrict__ in, int64_t n, unsigned long long* __restrict__ out) {
    __shared__ unsigned long long s_part[1024];
    const int64_t per = (n + 1023) / 1024;
    const int64_t lo = (int64_t)threadIdx.x * per, hi = lo + per < n ? lo + per : n;
    unsigned long long m = 0;
    for (int64_t t = lo; t < hi; ++t) m += in[t];
    s_part[threadIdx.x] = m;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const unsigned long long y = (int)threadIdx.x >= o ? s_part[threadIdx.x - o] : 0ull;
        __syncthreads();
        s_part[threadIdx.x] += y;
        __syncthreads();
    }
    unsigned long long run = threadIdx.x ? s_part[threadIdx.x - 1] : 0ull;
    for (int64_t t = lo; t < hi; ++t) {
        out[t] = run;
        run += in[t];
    }
    if (threadIdx.x == 1023) out[n] = s_part[1023];
}

__global__ void __launch_bounds__(PQ_THREADS) pq_str_write_kernel(const uint8_t* __restrict__ stage, const PqBlock* __restrict__ blocks, int64_t n_blocks,
                                                                 const uint64_t* __restrict__ row_ent, const unsigned long long* __restrict__ block_base,
                                                                 int32_t* __restrict__ offsets /* at the chunk's first row */, uint8_t* __restrict__ values,
                                                                 int64_t byte_base, int64_t num_values) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (PQ_THREADS / 32);
    for (int64_t b = (int64_t)blockIdx.x * (PQ_THREADS / 32) + (threadIdx.x >> 5); b < n_blocks; b += warps) {
        const PqBlock blk = blocks[b];
        unsigned long long running = (unsigned long long)byte_base + block_base[b];
        for (uint32_t i = 0; i < blk.n_rows; i += 32) {
            const bool in = i + lane < blk.n_rows;
            const uint64_t r = (uint64_t)blk.first_row + i + lane;
            const uint64_t ent = in ? row_ent[r] : 0ull;
            const uint32_t len = (uint32_t)(ent >> 40);
            uint32_t incl = len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            const unsigned long long start = running + incl - len;
            if (in) {
                offsets[r] = (int32_t)start;
                if (r + 1 == (uint64_t)num_values) offsets[r + 1] = (int32_t)(start + len);
                const uint8_t* src = stage + (ent & ((1ull << 40) - 1ull));
                uint8_t* dst = values + start;
                for (uint32_t k = 0; k < len; ++k) dst[k] = __ldg(src + k);
            }
            running += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
}

static void append_parquet_utf8(AppendTxn& txn, const std::string& name, int32_t max_def_level, int32_t codec, const uint8_t* chunk, int64_t n_bytes,
                                int64_t num_values) {
    Engine& e = txn.e;
    Column& c = txn.column(name, TG_UTF8);
    const int64_t have = c.n_rows;
    PqChunk pc;
    collect_sections(chunk, n_bytes, codec, max_def_level, num_values, TG_UTF8, pc);
    if (num_values == 0) return;
    const PqStaged st = stage_chunk(e, pc, PQ_KIND_STR, 0, max_def_level, num_values);
    std::vector<uint64_t> dict_ents;
    if (pc.dict_count > 0) {
        dict_ents.reserve((size_t)pc.dict_count);
        walk_plain_strings(pc.dict_values, pc.dict_bytes, pc.dict_count, (uint64_t)st.dict_off, dict_ents);
    }
    append_validity(e, c, have, st.bits.empty() ? nullptr : st.bits.data(), 0, num_values);

    // device tables: bits | blocks | runs | plain entries | dictionary entries | per-row entries | block totals | bases
    const int64_t nb = (int64_t)st.blocks.size();
    const std::vector<uint8_t*> d = upload_tables(e, st, num_values,
                                                  {{st.plain_ents.data(), st.plain_ents.size() * 8},
                                                   {dict_ents.data(), dict_ents.size() * 8},
                                                   {nullptr, (size_t)num_values * 8},
                                                   {nullptr, (size_t)(nb + 1) * 8},
                                                   {nullptr, (size_t)(nb + 1) * 8}});
    Utf8Entries x;
    x.stage = st.stage;
    x.blocks = reinterpret_cast<const PqBlock*>(d[1]);
    x.n_blocks = nb;
    x.row_ent = reinterpret_cast<const uint64_t*>(d[5]);
    x.block_bytes = reinterpret_cast<unsigned long long*>(d[6]);
    x.block_base = reinterpret_cast<unsigned long long*>(d[7]);
    pq_str_locate_kernel<<<pq_str_grid(e, nb), PQ_THREADS, 0, e.copy_stream>>>(
        st.stage, d[0], x.blocks, nb, reinterpret_cast<const PqRun*>(d[2]), reinterpret_cast<const uint64_t*>(d[3]),
        reinterpret_cast<const uint64_t*>(d[4]), (uint32_t)pc.dict_count, reinterpret_cast<uint64_t*>(d[5]), x.block_bytes);
    TG_CUDA(cudaGetLastError());
    e.launches += 1;
    append_utf8_from_entries(e, c, x, num_values);
}

uint32_t append_utf8_from_entries(Engine& e, Column& c, const Utf8Entries& x, int64_t num_values) {
    const int64_t have = c.n_rows, nb = x.n_blocks;
    const int grid = pq_str_grid(e, nb);
    pq_block_scan_kernel<<<1, 1024, 0, e.copy_stream>>>(x.block_bytes, nb, x.block_base);
    TG_CUDA(cudaGetLastError());
    e.launches += 1;
    unsigned long long total = 0;
    uint32_t err = 0;
    TG_CUDA(cudaMemcpyAsync(&total, x.block_base + nb, 8, cudaMemcpyDeviceToHost, e.copy_stream));
    if (x.err) TG_CUDA(cudaMemcpyAsync(&err, x.err, 4, cudaMemcpyDeviceToHost, e.copy_stream));
    TG_CUDA(cudaStreamSynchronize(e.copy_stream));  // the byte total decides the value buffer's size
    if (err) return err;
    if ((unsigned long long)c.value_bytes + total > (unsigned long long)INT32_MAX)
        throw Error(TG_ERR_UNSUPPORTED, "Utf8 column exceeds 2 GiB of value bytes (32-bit offsets)");
    e.dev_reserve(c.values, (size_t)(c.value_bytes + (int64_t)total), (size_t)c.value_bytes);
    e.dev_reserve(c.offsets, (size_t)(have + num_values + 1) * 4, have ? (size_t)(have + 1) * 4 : 0);
    pq_str_write_kernel<<<grid, PQ_THREADS, 0, e.copy_stream>>>(x.stage, x.blocks, nb, x.row_ent, x.block_base,
                                                               reinterpret_cast<int32_t*>(c.offsets.p) + have, c.values.p, c.value_bytes, num_values);
    TG_CUDA(cudaGetLastError());
    e.launches += 1;
    c.value_bytes += (int64_t)total;
    c.last_offset = (int32_t)c.value_bytes;
    c.n_rows = have + num_values;
    return 0;
}

// host-only (tests): one page's value section of a DELTA_* / BYTE_STREAM_SPLIT encoding rewritten to the PLAIN layout
int64_t parquet_decode_to_plain(int32_t encoding, int32_t elem_width, const uint8_t* src, int64_t n, int64_t n_values, uint8_t* dst, int64_t cap) {
    if (!src || n < 0 || n_values < 0 || (!dst && cap > 0) || cap < 0) throw Error(TG_ERR_INVALID_ARG, "NULL value buffers");
    if (elem_width != 0 && elem_width != 4 && elem_width != 8) throw Error(TG_ERR_INVALID_ARG, "element width must be 0 (BYTE_ARRAY), 4 or 8");
    std::vector<uint8_t> out;
    decode_to_plain(encoding, (size_t)elem_width, src, n, n_values, out);
    if ((int64_t)out.size() > cap) throw Error(TG_ERR_INVALID_ARG, "PLAIN rewrite larger than the output buffer");
    if (!out.empty()) memcpy(dst, out.data(), out.size());
    return (int64_t)out.size();
}

// host-only (tests): one page body through the codec dispatch of the chunk path
int64_t parquet_page_decompress(int32_t codec, const uint8_t* src, int64_t n, uint8_t* dst, int64_t cap) {
    if (!src || n < 0 || !dst || cap < 0) throw Error(TG_ERR_INVALID_ARG, "NULL page buffers");
    if (codec == PQ_CODEC_UNCOMPRESSED || !codec_supported(codec)) throw Error(TG_ERR_UNSUPPORTED, "Parquet: codec " + std::to_string(codec) + " has no decoder");
    return (int64_t)page_decompress(codec, src, (size_t)n, dst, (size_t)cap);
}

// host-only (tests): Snappy raw-format decompression as the Parquet path uses it; returns the uncompressed size
int64_t parquet_snappy_decompress(const uint8_t* src, int64_t n, uint8_t* dst, int64_t cap) {
    if (!src || n <= 0 || !dst || cap < 0) throw Error(TG_ERR_INVALID_ARG, "NULL Snappy buffers");
    return (int64_t)snappy_decompress(src, (size_t)n, dst, (size_t)cap);
}

}  // namespace tg
