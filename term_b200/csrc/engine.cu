// Engine: device memory, Arrow buffer marshalling (pinned double-buffered H2D), job dispatch, and the
// planner of the fused numeric scan (which units run on which consumer warp of scan_kernel).
#include "engine.hpp"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <ctime>

namespace tg {

constexpr size_t PINNED_CHUNK = 32u << 20;
constexpr size_t PAD = 256;

static size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

uint8_t* Engine::scratch(size_t bytes) {
    if (bytes > scratch_cap) {
        TG_CUDA(cudaStreamSynchronize(stream));
        if (d_scratch) TG_CUDA(cudaFree(d_scratch));
        scratch_cap = round_up(std::max(bytes, (size_t)1 << 20), 1 << 20);
        TG_CUDA(cudaMalloc(&d_scratch, scratch_cap));
    }
    return d_scratch;
}

void Engine::ensure_side_streams() {
    if (side[0]) return;
    for (auto& s : side) TG_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    for (auto& ev : side_ev) TG_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
}

uint8_t* Engine::aux(size_t bytes) {
    if (bytes > aux_cap) {
        TG_CUDA(cudaStreamSynchronize(stream));
        if (d_aux) TG_CUDA(cudaFree(d_aux));
        d_aux = nullptr;
        aux_cap = 0;
        const size_t ncap = round_up(std::max(bytes, (size_t)1 << 20), 1 << 20);
        TG_CUDA(cudaMalloc(&d_aux, ncap));
        aux_cap = ncap;
    }
    return d_aux;
}

uint8_t* Engine::host_scratch(size_t bytes) {
    if (bytes > h_scratch_cap) {
        if (h_scratch) TG_CUDA(cudaFreeHost(h_scratch));
        h_scratch_cap = round_up(std::max(bytes, (size_t)1 << 16), 1 << 16);
        TG_CUDA(cudaMallocHost(&h_scratch, h_scratch_cap));
    }
    return h_scratch;
}

// Device blocks of tables are recycled through an exact-size free list: registering a table of the same shape
// again (the steady state of a validation service, and of bench.py's end-to-end loop) costs no cudaMalloc /
// cudaFree, which for multi-GB buffers are milliseconds each and serialise the device.
uint8_t* Engine::dev_alloc(size_t bytes) {
    auto it = free_blocks.find(bytes);
    if (it != free_blocks.end() && !it->second.empty()) {
        uint8_t* p = it->second.back();
        it->second.pop_back();
        cached_bytes -= bytes;
        return p;
    }
    uint8_t* p = nullptr;
    cudaError_t err = cudaMalloc(&p, bytes);
    if (err != cudaSuccess) {
        cudaGetLastError();
        dev_trim();
        TG_CUDA(cudaMalloc(&p, bytes));
    }
    return p;
}
void Engine::dev_free(uint8_t* p, size_t bytes) {
    if (!p) return;
    if (bytes == 0 || cached_bytes + bytes > cache_limit) {
        cudaFree(p);
        return;
    }
    free_blocks[bytes].push_back(p);
    cached_bytes += bytes;
}
void Engine::dev_trim() {
    for (auto& kv : free_blocks)
        for (uint8_t* p : kv.second) cudaFree(p);
    free_blocks.clear();
    cached_bytes = 0;
}

// grow a device buffer to hold `need` bytes (+ zeroed padding), preserving the first keep_bytes
void Engine::dev_reserve(DevBuf& b, size_t need, size_t keep_bytes) {
    const size_t padded = round_up(need + PAD, PAD);
    if (!(b.p && padded <= b.cap)) {
        size_t ncap = b.p ? std::max(padded, b.cap + b.cap / 2) : padded;
        ncap = round_up(ncap, PAD);
        uint8_t* np = dev_alloc(ncap);
        if (b.p && keep_bytes) TG_CUDA(cudaMemcpyAsync(np, b.p, keep_bytes, cudaMemcpyDeviceToDevice, copy_stream));
        if (b.p) {
            TG_CUDA(cudaStreamSynchronize(copy_stream));
            TG_CUDA(cudaStreamSynchronize(stream));
            if (b.owned) dev_free(b.p, b.cap);
        }
        b.p = np;
        b.cap = ncap;
        b.owned = true;
    }
    // zero the padding behind the new logical end (kernels over-read it with TMA / 128-bit loads)
    TG_CUDA(cudaMemsetAsync(b.p + need, 0, padded - need, copy_stream));
}

void Engine::h2d(void* dst, const void* src, size_t bytes, cudaStream_t s) {
    if (bytes == 0) return;
    if (!s) s = copy_stream;
    cudaPointerAttributes attr{};
    bool pinned_src = false;
    if (cudaPointerGetAttributes(&attr, src) == cudaSuccess) pinned_src = attr.type == cudaMemoryTypeHost;
    else cudaGetLastError();
    if (pinned_src) {
        TG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s));
        return;
    }
    // pageable source: stage through the pinned ring so the CPU memcpy of chunk i+1 overlaps the DMA of chunk i
    size_t off = 0;
    while (off < bytes) {
        size_t n = std::min(PINNED_CHUNK, bytes - off);
        int k = pinned_next;
        pinned_next ^= 1;
        TG_CUDA(cudaEventSynchronize(pinned_free[k]));
        memcpy(pinned[k], (const uint8_t*)src + off, n);
        TG_CUDA(cudaMemcpyAsync((uint8_t*)dst + off, pinned[k], n, cudaMemcpyHostToDevice, s));
        TG_CUDA(cudaEventRecord(pinned_free[k], s));
        off += n;
    }
}

void Engine::sync_copies() {
    TG_CUDA(cudaStreamSynchronize(copy_stream));
    for (auto& b : deferred_free) dev_free(b.first, b.second);
    deferred_free.clear();
}

// ------------------------------------------------------------------ scan planning ----

struct ScanOp {
    int kind;  // UNIT_*
    int agg;
    Column* c0 = nullptr;
    Column* c1 = nullptr;
    double cost = 1.0;
    int flags = 0;
    std::vector<PredInstr> code;
    std::vector<ScanTerm> terms;
    std::vector<Column*> pred_cols;
};

struct TileCol {
    Column* col;
    bool need_values;
};

static int tile_col_index(std::vector<TileCol>& tc, Column* c, bool need_values) {
    for (size_t i = 0; i < tc.size(); ++i)
        if (tc[i].col == c) {
            tc[i].need_values |= need_values;
            return (int)i;
        }
    tc.push_back(TileCol{c, need_values});
    return (int)tc.size() - 1;
}

static std::string no_field_msg(const Table& t, const std::string& col) {
    return "Schema error: No field named " + col + ". Valid fields are " + t.valid_fields() + ".";
}

__global__ void scan_states_kernel(const ScanAggOut* __restrict__ out, const ScanOpMeta* __restrict__ metas, int n_ops, DevAggRec* __restrict__ states);

static void run_scan_pass(Engine& e, Table& t, Plan& p, std::vector<ScanOp>& ops) {
    if (ops.empty()) return;
    auto P = std::make_unique<ScanParams>();
    memset(P.get(), 0, sizeof(ScanParams));
    std::vector<TileCol> tcols;
    // tile columns
    struct OpCols {
        int c0 = -1, c1 = -1;
    };
    std::vector<OpCols> oc(ops.size());
    for (size_t i = 0; i < ops.size(); ++i) {
        ScanOp& o = ops[i];
        if (o.kind == UNIT_COUNT) oc[i].c0 = tile_col_index(tcols, o.c0, false);
        else if (o.kind == UNIT_NUM_F64 || o.kind == UNIT_NUM_I64) oc[i].c0 = tile_col_index(tcols, o.c0, true);
        else if (o.kind == UNIT_PAIR) {
            oc[i].c0 = tile_col_index(tcols, o.c0, true);
            oc[i].c1 = tile_col_index(tcols, o.c1, true);
        } else if (o.kind == UNIT_PRED || o.kind == UNIT_TERMS) {
            for (size_t k = 0; k < o.pred_cols.size(); ++k) {
                bool need_values = true;
                if (o.kind == UNIT_TERMS) {  // IS [NOT] NULL terms only need the validity bitmap
                    need_values = false;
                    for (auto& tm : o.terms)
                        if (tm.col == (int)k && tm.kind != TK_ISNULL && tm.kind != TK_NOTNULL) need_values = true;
                }
                tile_col_index(tcols, o.pred_cols[k], need_values);
            }
        }
    }
    if (tcols.size() > (size_t)SCAN_MAX_COLS) throw Error(TG_ERR_UNSUPPORTED, "too many columns in one scan pass");
    // predicate code was compiled against per-op column order; remap to tile indices
    int code_len_total = 0;
    for (auto& o : ops) code_len_total += (int)o.code.size();
    if (code_len_total > SCAN_MAX_CODE) throw Error(TG_ERR_UNSUPPORTED, "predicates too long for one scan pass");

    // bytes per row -> tile rows / stages
    auto stage_bytes_for = [&](int tile_rows, std::vector<uint32_t>* val_off, std::vector<uint32_t>* bit_off) {
        size_t off = 0;
        for (size_t i = 0; i < tcols.size(); ++i) {
            if (tcols[i].need_values) {
                if (val_off) (*val_off)[i] = (uint32_t)off;
                size_t b = tcols[i].col->dtype == TG_BOOL ? (size_t)tile_rows / 8 : (size_t)tile_rows * 8;
                off += round_up(b, 128);
            }
            if (tcols[i].col->validity.p) {
                if (bit_off) (*bit_off)[i] = (uint32_t)off;
                off += round_up((size_t)tile_rows / 8, 128);
            }
        }
        return off;
    };
    // units: ops are replicated over row slices of the tile (multiples of 128 rows) so that every consumer warp
    // owns one unit of similar cost and keeps it in registers; warps are handed out greedily to the op whose
    // per-replica cost is largest
    int tile_rows = 4096;
    if (const char* ev = getenv("TG_SCAN_TILE_ROWS")) tile_rows = std::max(128, atoi(ev) / 128 * 128);
    int min_stages = 3;
    if (const char* ev = getenv("TG_SCAN_MIN_STAGES")) min_stages = std::max(2, atoi(ev));
    // units to aim for: one per consumer warp keeps every unit's state in registers; a plan with more aggregates
    // than warps already pays for shared-memory state, so it is split finer (better LPT balance)
    int target_units = SCAN_CONSUMER_WARPS;
    if (const char* ev = getenv("TG_SCAN_UNITS")) target_units = std::min(SCAN_MAX_UNITS, std::max(1, atoi(ev)));
    int n_stages = 0;
    std::vector<int> reps(ops.size(), 1);
    size_t stage_bytes = 0, state_bytes = 0;
    const size_t smem_budget = 227 * 1024 - 256 - sizeof(ScanTables);
    for (; tile_rows >= 128; tile_rows /= 2) {
        const int chunks = tile_rows / 128;
        int n_units = (int)ops.size();
        for (size_t i = 0; i < ops.size(); ++i) reps[i] = 1;
        while (n_units < target_units) {
            int best = -1;
            double best_cost = 0;
            for (size_t i = 0; i < ops.size(); ++i) {
                if (ops[i].kind == UNIT_COUNT || reps[i] >= chunks) continue;
                const double c = ops[i].cost / reps[i];
                if (c > best_cost) {
                    best_cost = c;
                    best = (int)i;
                }
            }
            if (best < 0) break;
            ++reps[best];
            ++n_units;
        }
        if (n_units > SCAN_MAX_UNITS) throw Error(TG_ERR_UNSUPPORTED, "too many aggregates in one scan pass");
        state_bytes = n_units <= SCAN_CONSUMER_WARPS ? 0 : (size_t)n_units * SCAN_STATE_SLOTS * 32 * 8;
        stage_bytes = stage_bytes_for(tile_rows, nullptr, nullptr);
        if (stage_bytes == 0) stage_bytes = 128;
        if (state_bytes + (size_t)min_stages * stage_bytes + 2 * SCAN_MAX_STAGES * 8 <= smem_budget) {
            n_stages = (int)std::min<size_t>(SCAN_MAX_STAGES, (smem_budget - state_bytes - 2 * SCAN_MAX_STAGES * 8) / stage_bytes);
            break;
        }
    }
    if (n_stages < 2) throw Error(TG_ERR_UNSUPPORTED, "scan pass does not fit in shared memory");

    std::vector<uint32_t> val_off(tcols.size(), 0), bit_off(tcols.size(), 0);
    stage_bytes_for(tile_rows, &val_off, &bit_off);
    P->n_rows = t.n_rows;
    P->tile_rows = tile_rows;
    P->n_tiles = (t.n_rows + tile_rows - 1) / tile_rows;
    P->n_cols = (int)tcols.size();
    P->n_stages = n_stages;
    P->stage_bytes = (uint32_t)stage_bytes;
    for (size_t i = 0; i < tcols.size(); ++i) {
        Column* c = tcols[i].col;
        ScanColDesc& d = P->tab.cols[i];
        d.values = tcols[i].need_values ? c->values.p : nullptr;
        d.validity = c->validity.p;
        d.kind = c->dtype == TG_FLOAT64 ? SC_F64 : c->dtype == TG_INT64 ? SC_I64 : c->dtype == TG_BOOL ? SC_BOOL : SC_BITS;
        if (!tcols[i].need_values) d.kind = SC_BITS;
        d.smem_val_off = val_off[i];
        d.smem_bits_off = bit_off[i];
        d.pivot = c->pivot;
        d.ipivot = c->ipivot;
        d.pivot_is_element = c->pivot_set ? 1 : 0;
    }
    // units + code / terms
    int term_off = 0;
    struct UnitTmp {
        ScanUnitDesc d;
        double cost;
    };
    std::vector<UnitTmp> units;
    int code_off = 0;
    for (size_t i = 0; i < ops.size(); ++i) {
        ScanOp& o = ops[i];
        int this_code_off = code_off;
        if (o.kind == UNIT_PRED) {
            for (auto ins : o.code) {
                // operands referencing columns carry an index into o.pred_cols; translate to tile columns
                auto fix = [&](uint8_t kind, uint16_t& idx) {
                    if (kind == PK_COL_F64 || kind == PK_COL_I64 || kind == PK_COL_I64_AS_F64 || kind == PK_COL_BOOL)
                        idx = (uint16_t)tile_col_index(tcols, o.pred_cols[idx], true);
                };
                fix(ins.a_kind, ins.a_idx);
                fix(ins.b_kind, ins.b_idx);
                P->tab.code[code_off++] = ins;
            }
        }
        if (o.kind == UNIT_TERMS) {
            this_code_off = term_off;
            for (auto tm : o.terms) {
                tm.col = tile_col_index(tcols, o.pred_cols[tm.col], false);
                if (term_off >= SCAN_MAX_TERMS) throw Error(TG_ERR_UNSUPPORTED, "too many predicate terms in one scan pass");
                P->tab.terms[term_off++] = tm;
            }
        }
        const int r = reps[i];
        const int chunks = tile_rows / 128;
        for (int k = 0; k < r; ++k) {
            UnitTmp u{};
            u.d.kind = o.kind;
            u.d.c0 = oc[i].c0;
            u.d.c1 = oc[i].c1;
            u.d.row0 = (k * chunks / r) * 128;
            u.d.nrows = ((k + 1) * chunks / r) * 128 - u.d.row0;
            u.d.agg = (int)i;  // local aggregate index within this pass
            u.d.code_off = this_code_off;
            u.d.code_len = o.kind == UNIT_TERMS ? (int)o.terms.size() : (int)o.code.size();
            u.d.c0_is_i64 = o.c0 && o.c0->dtype == TG_INT64;
            u.d.c1_is_i64 = o.c1 && o.c1->dtype == TG_INT64;
            u.d.flags = o.flags;
            u.cost = o.cost * u.d.nrows / tile_rows;
            units.push_back(u);
        }
    }
    // LPT assignment of units to consumer warps
    std::vector<int> order(units.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return units[a].cost > units[b].cost; });
    double load[SCAN_CONSUMER_WARPS] = {0};
    int owned[SCAN_CONSUMER_WARPS] = {0};
    for (int idx : order) {
        int best = -1;
        for (int w = 0; w < SCAN_CONSUMER_WARPS; ++w)
            if (owned[w] < SCAN_WARP_UNITS && (best < 0 || load[w] < load[best])) best = w;
        if (best < 0) throw Error(TG_ERR_UNSUPPORTED, "too many aggregates in one scan pass");
        units[idx].d.warp = best;
        load[best] += units[idx].cost;
        P->tab.warp_units[best][1 + owned[best]] = idx;
        P->tab.warp_units[best][0] = ++owned[best];
    }
    P->n_units = (int)units.size();
    P->n_state_units = units.size() <= (size_t)SCAN_CONSUMER_WARPS ? 0 : (int)units.size();
    P->n_aggs = (int)ops.size();
    P->n_code = code_off;
    P->n_terms = term_off;
    for (size_t i = 0; i < units.size(); ++i) P->tab.units[i] = units[i].d;

    const int grid = (int)std::min<int64_t>(std::max<int64_t>(P->n_tiles, 1), e.sm_count);
    const size_t partial_bytes = (size_t)grid * P->n_units * SCAN_STATE_SLOTS * 8;
    const size_t out_bytes = ops.size() * sizeof(ScanAggOut);
    uint8_t* scr = e.scratch(round_up(partial_bytes, 256) + out_bytes);
    P->partials = reinterpret_cast<uint64_t*>(scr);
    ScanAggOut* d_out = reinterpret_cast<ScanAggOut*>(scr + round_up(partial_bytes, 256));

    TG_CUDA(cudaEventRecord(e.ev[0], e.stream));
    TG_CUDA(scan_launch(*P, grid, d_out, e.stream));
    TG_CUDA(cudaEventRecord(e.ev[1], e.stream));
    e.launches += 2;
    p.stats.launches += 2;
    if (e.fused) {
        // fused multi-GPU step: no copy-out, no synchronisation — a small kernel turns the records into partial states
        // on the device (the decode below, restated in scan_states_kernel)
        FusedScan& fz = *e.fused;
        ScanOpMeta* hm = fz.h_metas + fz.n_metas;
        for (size_t i = 0; i < ops.size(); ++i) {
            hm[i] = ScanOpMeta{ops[i].kind, ops[i].agg, ops[i].c0 ? ops[i].c0->pivot : 0.0, ops[i].c1 ? ops[i].c1->pivot : 0.0, (uint64_t)t.n_rows};
            fz.from_device[ops[i].agg] = 1;
        }
        // the few bytes of per-op metadata are read by the kernel straight from pinned host memory (UVA): no copy call
        scan_states_kernel<<<1, 64, 0, e.stream>>>(d_out, hm, (int)ops.size(), fz.d_states);
        TG_CUDA(cudaGetLastError());
        fz.n_metas += (int)ops.size();
        e.launches += 1;
        p.stats.launches += 1;
        return;
    }
    ScanAggOut* h_out = reinterpret_cast<ScanAggOut*>(e.host_scratch(out_bytes));
    TG_CUDA(cudaMemcpyAsync(h_out, d_out, out_bytes, cudaMemcpyDeviceToHost, e.stream));
    TG_CUDA(cudaStreamSynchronize(e.stream));
    float ms = 0;
    TG_CUDA(cudaEventElapsedTime(&ms, e.ev[0], e.ev[1]));
    p.stats.scan_ms += ms;
    p.stats.gpu_ms += ms;

    auto u2d = [](uint64_t u) {
        double d;
        memcpy(&d, &u, 8);
        return d;
    };
    for (size_t i = 0; i < ops.size(); ++i) {
        Agg& a = p.aggs[ops[i].agg];
        const uint64_t* s = h_out[i].s;
        switch (ops[i].kind) {
            case UNIT_COUNT:
                a.u[0] = (uint64_t)t.n_rows;
                a.u[1] = s[S_N];
                break;
            case UNIT_NUM_F64:
            case UNIT_NUM_I64:
                a.u[0] = s[S_N];
                a.f[0] = ops[i].c0->pivot;
                a.f[1] = u2d(s[S_SD]);
                a.f[2] = u2d(s[S_SDD]);
                a.f[5] = (double)s[S_N] * ops[i].c0->pivot + u2d(s[S_SD]);  // sum(x) = n*K + sum(x-K)
                if (ops[i].kind == UNIT_NUM_I64) {
                    a.u[1] = s[S_ISUM];  // wrapping i64 sum over the valid rows
                    a.u[2] = s[S_MIN];
                    a.u[3] = s[S_MAX];
                    a.u[4] = 1;
                } else {
                    a.f[3] = u2d(s[S_MIN]);
                    a.f[4] = u2d(s[S_MAX]);
                }
                break;
            case UNIT_PAIR:
                a.u[0] = s[P_N];
                a.f[0] = ops[i].c0->pivot;
                a.f[1] = ops[i].c1->pivot;
                a.f[2] = u2d(s[P_SX]);
                a.f[3] = u2d(s[P_SY]);
                a.f[4] = u2d(s[P_SXX]);
                a.f[5] = u2d(s[P_SYY]);
                a.f[6] = u2d(s[P_SXY]);
                break;
            case UNIT_PRED:
            case UNIT_TERMS:
                a.u[0] = s[0];
                a.u[1] = ops[i].kind == UNIT_PRED ? s[1] : 0;
                a.u[2] = (uint64_t)t.n_rows;
                break;
        }
    }
}

// the decode above on the device (fused multi-GPU step): record i of a pass -> the partial state of its aggregate
__global__ void scan_states_kernel(const ScanAggOut* __restrict__ out, const ScanOpMeta* __restrict__ metas, int n_ops, DevAggRec* __restrict__ states) {
    for (int i = threadIdx.x; i < n_ops; i += blockDim.x) {
        const ScanOpMeta m = metas[i];
        const uint64_t* s = out[i].s;
        DevAggRec& a = states[m.agg];
        auto u2d = [](uint64_t u) { return __longlong_as_double((long long)u); };
        switch (m.unit_kind) {
            case UNIT_COUNT:
                a.u[0] = m.n_rows;
                a.u[1] = s[S_N];
                break;
            case UNIT_NUM_F64:
            case UNIT_NUM_I64:
                a.u[0] = s[S_N];
                a.f[0] = m.pivot0;
                a.f[1] = u2d(s[S_SD]);
                a.f[2] = u2d(s[S_SDD]);
                a.f[5] = __dadd_rn(__dmul_rn((double)s[S_N], m.pivot0), u2d(s[S_SD]));  // as the host: product and sum rounded separately
                if (m.unit_kind == UNIT_NUM_I64) {
                    a.u[1] = s[S_ISUM];
                    a.u[2] = s[S_MIN];
                    a.u[3] = s[S_MAX];
                    a.u[4] = 1;
                } else {
                    a.f[3] = u2d(s[S_MIN]);
                    a.f[4] = u2d(s[S_MAX]);
                }
                break;
            case UNIT_PAIR:
                a.u[0] = s[P_N];
                a.f[0] = m.pivot0;
                a.f[1] = m.pivot1;
                a.f[2] = u2d(s[P_SX]);
                a.f[3] = u2d(s[P_SY]);
                a.f[4] = u2d(s[P_SXX]);
                a.f[5] = u2d(s[P_SYY]);
                a.f[6] = u2d(s[P_SXY]);
                break;
            default:  // UNIT_PRED / UNIT_TERMS
                a.u[0] = s[0];
                a.u[1] = m.unit_kind == UNIT_PRED ? s[1] : 0;
                a.u[2] = m.n_rows;
                break;
        }
    }
}

// the rank's payload for the mailbox: [u64 byte length][u64 n_aggs][n_aggs x DevAggRec] from the host's template (aggregates
// the host resolved, error codes) and the device states; COUNT(c) aggregates folded into a NUM unit take its count
__global__ void scan_payload_kernel(const DevAggRec* __restrict__ tmpl, const uint8_t* __restrict__ from_device, const DevAggRec* __restrict__ states,
                                    const int2* __restrict__ folds, int n_folds, int n_aggs, uint64_t n_rows, uint8_t* __restrict__ payload) {
    uint64_t* hdr = reinterpret_cast<uint64_t*>(payload);
    DevAggRec* recs = reinterpret_cast<DevAggRec*>(payload + 16);
    for (int i = threadIdx.x; i < n_aggs; i += blockDim.x) {
        DevAggRec r = tmpl[i];
        if (from_device[i]) {
            const DevAggRec s = states[i];
            for (int k = 0; k < 8; ++k) {
                r.u[k] = s.u[k];
                r.f[k] = s.f[k];
            }
        }
        recs[i] = r;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_folds; i += blockDim.x) {
        recs[folds[i].x].u[0] = n_rows;
        recs[folds[i].x].u[1] = recs[folds[i].y].u[0];
    }
    if (threadIdx.x == 0) {
        hdr[0] = 8 + (uint64_t)n_aggs * sizeof(DevAggRec);
        hdr[1] = (uint64_t)n_aggs;
    }
}

// ---- string-literal comparisons inside predicates --------------------------------------------------
// `utf8_col = 'lit'` / `<>` (and IN lists, which desugar to them) are materialised by a small kernel into a
// bit-packed BOOLEAN virtual column (validity = the string column's validity) that the fused scan then
// reads like any other column; e.g. `status = 'active' AND price >= 10` (constraints/custom_sql.rs:440-456).
__global__ void str_eq_kernel(const int32_t* offsets, const uint8_t* bytes, int64_t n, const uint8_t* lit, int32_t lit_len,
                              uint32_t* out_bits) {
    for (int64_t base = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) & ~31ll; base < n;
         base += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = base + (threadIdx.x & 31);
        bool eq = false;
        if (row < n) {
            const int32_t b = offsets[row], e = offsets[row + 1];
            eq = (e - b) == lit_len;
            for (int32_t k = 0; eq && k < lit_len; ++k) eq = bytes[b + k] == lit[k];
        }
        const uint32_t w = __ballot_sync(0xffffffffu, eq);
        if ((threadIdx.x & 31) == 0) out_bits[base >> 5] = w;
    }
}

// ---- Int32 / Float32 columns ------------------------------------------------------------------------
// SUM / AVG / STDDEV / CORR and predicates over a 4-byte column are defined by DataFusion on the value widened to Int64 /
// Float64 (both exact), so the 8-byte kernels serve them through a widened shadow column: values converted on the device
// (the 4-byte data crossed PCIe once), validity shared with the source column.
__global__ void widen_kernel(const uint32_t* __restrict__ src, uint64_t* __restrict__ dst, int64_t n, int is_float) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t v = __ldg(src + i);
        dst[i] = is_float ? (uint64_t)__double_as_longlong((double)__uint_as_float(v)) : (uint64_t)(int64_t)(int32_t)v;
    }
}

Column* numeric_view(Engine& e, Column* c) {
    if (!c) return nullptr;
    if (c->dtype == TG_INT64 || c->dtype == TG_FLOAT64) return c;
    if (c->dtype != TG_INT32 && c->dtype != TG_FLOAT32) return nullptr;
    if (!c->wide) c->wide = std::make_unique<Column>();
    Column& w = *c->wide;
    if (w.n_rows != c->n_rows || !w.values.p) {
        e.sync_copies();  // the 4-byte values may still be in flight on the copy stream
        w.name = c->name;
        w.dtype = c->dtype == TG_INT32 ? TG_INT64 : TG_FLOAT64;
        e.dev_reserve(w.values, (size_t)c->n_rows * 8, 0);
        if (c->n_rows > 0) {
            const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((c->n_rows + 255) / 256, (int64_t)e.sm_count * 16));
            widen_kernel<<<grid, 256, 0, e.stream>>>(reinterpret_cast<const uint32_t*>(c->values.p), reinterpret_cast<uint64_t*>(w.values.p),
                                                     c->n_rows, c->dtype == TG_FLOAT32 ? 1 : 0);
            TG_CUDA(cudaGetLastError());
            e.launches += 1;
            // pivot of the shifted sums: from the first values, like every 8-byte column
            const int64_t head = std::min<int64_t>(c->n_rows, 65536);
            std::vector<uint8_t> hv((size_t)head * 8), hb((size_t)(head + 7) / 8);
            TG_CUDA(cudaMemcpyAsync(hv.data(), w.values.p, hv.size(), cudaMemcpyDeviceToHost, e.stream));
            if (c->validity.p) TG_CUDA(cudaMemcpyAsync(hb.data(), c->validity.p, hb.size(), cudaMemcpyDeviceToHost, e.stream));
            TG_CUDA(cudaStreamSynchronize(e.stream));
            w.pivot_set = false;
            set_pivot_host(w, w.dtype, head, hv.data(), c->validity.p ? hb.data() : nullptr, 0);
        }
        w.n_rows = c->n_rows;
        w.value_bytes = c->n_rows * 8;
    }
    w.validity.p = c->validity.p;  // (may have been reallocated by an append: refreshed on every use)
    w.validity.cap = 0;
    w.validity.owned = false;
    w.null_count = c->null_count;
    return &w;
}

void column_free(Engine& e, Column& c) {
    if (c.values.owned && c.values.p) e.dev_free(c.values.p, c.values.cap);
    if (c.offsets.owned && c.offsets.p) e.dev_free(c.offsets.p, c.offsets.cap);
    if (c.validity.owned && c.validity.p) e.dev_free(c.validity.p, c.validity.cap);
    if (c.wide && c.wide->values.owned && c.wide->values.p) e.dev_free(c.wide->values.p, c.wide->values.cap);
    c.wide.reset();
}

struct VirtualCols {
    Engine& e;
    std::vector<std::unique_ptr<Column>> cols;
    explicit VirtualCols(Engine& e_) : e(e_) {}
    ~VirtualCols() {
        cudaStreamSynchronize(e.stream);
        for (auto& c : cols)
            if (c->values.p) cudaFree(c->values.p);
    }
};

// ---- the other string sub-expressions of a predicate, materialised the same way ----
// comparisons (byte-wise, the order DataFusion gives Utf8: UTF-8 preserves code-point order) of a Utf8 column with a
// literal or with another Utf8 column; op: 0 =, 1 <>, 2 <, 3 <=, 4 >, 5 >=. out_valid (column-column only) = both valid.
__device__ __forceinline__ int str_bytes_cmp(const uint8_t* a, int32_t la, const uint8_t* b, int32_t lb) {
    const int32_t m = la < lb ? la : lb;
    for (int32_t k = 0; k < m; ++k)
        if (a[k] != b[k]) return a[k] < b[k] ? -1 : 1;
    return la < lb ? -1 : (la > lb ? 1 : 0);
}
__global__ void str_cmp_kernel(const int32_t* offs_a, const uint8_t* bytes_a, const int32_t* offs_b, const uint8_t* bytes_b, int32_t lit_len,
                               const uint32_t* valid_a, const uint32_t* valid_b, int64_t n, int op, uint32_t* out_bits, uint32_t* out_valid) {
    for (int64_t base = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) & ~31ll; base < n; base += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = base + (threadIdx.x & 31);
        bool r = false;
        if (row < n) {
            const int32_t a0 = offs_a[row], a1 = offs_a[row + 1];
            const uint8_t* pb = bytes_b;
            int32_t lb = lit_len;
            if (offs_b) {
                pb = bytes_b + offs_b[row];
                lb = offs_b[row + 1] - offs_b[row];
            }
            const int c = str_bytes_cmp(bytes_a + a0, a1 - a0, pb, lb);
            r = op == 0 ? c == 0 : op == 1 ? c != 0 : op == 2 ? c < 0 : op == 3 ? c <= 0 : op == 4 ? c > 0 : c >= 0;
        }
        const uint32_t w = __ballot_sync(0xffffffffu, r);
        if ((threadIdx.x & 31) == 0) {
            out_bits[base >> 5] = w;
            if (out_valid) out_valid[base >> 5] = (valid_a ? valid_a[base >> 5] : 0xffffffffu) & (valid_b ? valid_b[base >> 5] : 0xffffffffu);
        }
    }
}
// LENGTH / CHAR_LENGTH / CHARACTER_LENGTH (characters: bytes that are not UTF-8 continuation bytes) and OCTET_LENGTH
__global__ void str_length_kernel(const int32_t* offsets, const uint8_t* bytes, int64_t n, int octets, int64_t* out) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x) {
        const int32_t b = offsets[row], e = offsets[row + 1];
        int64_t c = e - b;
        if (!octets) {
            c = 0;
            for (int32_t k = b; k < e; ++k) c += (bytes[k] & 0xC0) != 0x80;
        }
        out[row] = c;
    }
}
// LIKE: the pattern as tokens (kind 0: this byte, 1: `_` one character, 2: `%` any sequence); greedy match with
// backtracking to the last `%`, stepping whole UTF-8 characters
__global__ void str_like_kernel(const int32_t* offsets, const uint8_t* bytes, int64_t n, const uint8_t* tok_kind, const uint8_t* tok_byte, int32_t m,
                                uint32_t* out_bits) {
    for (int64_t base = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) & ~31ll; base < n; base += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = base + (threadIdx.x & 31);
        bool ok = false;
        if (row < n) {
            const uint8_t* str = bytes + offsets[row];
            const int32_t len = offsets[row + 1] - offsets[row];
            auto next_char = [&](int32_t i) {
                ++i;
                while (i < len && (str[i] & 0xC0) == 0x80) ++i;
                return i;
            };
            int32_t si = 0, pi = 0, star_p = -1, star_s = 0;
            bool fail = false;
            while (si < len) {
                if (pi < m && tok_kind[pi] == 0 && str[si] == tok_byte[pi]) {
                    ++si;
                    ++pi;
                } else if (pi < m && tok_kind[pi] == 1) {
                    si = next_char(si);
                    ++pi;
                } else if (pi < m && tok_kind[pi] == 2) {
                    star_p = pi++;
                    star_s = si;
                } else if (star_p >= 0) {
                    pi = star_p + 1;
                    star_s = next_char(star_s);
                    si = star_s;
                } else {
                    fail = true;
                    break;
                }
            }
            while (!fail && pi < m && tok_kind[pi] == 2) ++pi;
            ok = !fail && pi == m;
        }
        const uint32_t w = __ballot_sync(0xffffffffu, ok);
        if ((threadIdx.x & 31) == 0) out_bits[base >> 5] = w;
    }
}

// ---- date / timestamp literals ----------------------------------------------------------------------
// `date_col >= '2024-01-31'`, `ts_col < '2024-01-31 10:11:12.5'` (also with a T separator, Z / +hh:mm offsets and the typed forms
// DATE '..' / TIMESTAMP '..'): DataFusion casts the string to the column's type; here the literal becomes the column's integer
// (days for Date32, the timestamp unit otherwise; naive literals are UTC). Returns false when the text is not a date / timestamp.
static int64_t days_from_civil(int64_t y, unsigned m, unsigned d) {  // proleptic Gregorian, days since 1970-01-01
    y -= m <= 2;
    const int64_t era = (y >= 0 ? y : y - 399) / 400;
    const unsigned yoe = (unsigned)(y - era * 400);
    const unsigned doy = (153 * (m + (m > 2 ? -3 : 9)) + 2) / 5 + d - 1;
    const unsigned doe = yoe * 365 + yoe / 4 - yoe / 100 + doy;
    return era * 146097 + (int64_t)doe - 719468;
}
static bool parse_temporal_literal(const std::string& text, char unit, int64_t* out) {
    size_t i = 0;
    auto digits = [&](int n, int64_t* v) {
        if (i + (size_t)n > text.size()) return false;
        int64_t x = 0;
        for (int k = 0; k < n; ++k) {
            if (!isdigit((unsigned char)text[i + k])) return false;
            x = x * 10 + (text[i + k] - '0');
        }
        i += (size_t)n;
        *v = x;
        return true;
    };
    int64_t Y, M, D, h = 0, mi = 0, sec = 0, frac_ns = 0, off_s = 0;
    if (!digits(4, &Y) || i >= text.size() || text[i++] != '-' || !digits(2, &M) || i >= text.size() || text[i++] != '-' || !digits(2, &D)) return false;
    static const int mdays[12] = {31, 29, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31};
    if (M < 1 || M > 12 || D < 1 || D > mdays[M - 1]) return false;
    if (M == 2 && D == 29 && !((Y % 4 == 0 && Y % 100 != 0) || Y % 400 == 0)) return false;
    bool has_time = false;
    if (i < text.size()) {
        if (text[i] != ' ' && text[i] != 'T' && text[i] != 't') return false;
        ++i;
        has_time = true;
        if (!digits(2, &h) || i >= text.size() || text[i++] != ':' || !digits(2, &mi)) return false;
        if (i < text.size() && text[i] == ':') {
            ++i;
            if (!digits(2, &sec)) return false;
            if (i < text.size() && text[i] == '.') {
                ++i;
                int n = 0;
                int64_t f = 0;
                while (i < text.size() && isdigit((unsigned char)text[i])) {
                    if (n < 9) {
                        f = f * 10 + (text[i] - '0');
                        ++n;
                    }
                    ++i;
                }
                if (n == 0) return false;
                while (n++ < 9) f *= 10;
                frac_ns = f;
            }
        }
        if (h > 23 || mi > 59 || sec > 59) return false;
        if (i < text.size() && (text[i] == 'Z' || text[i] == 'z')) ++i;
        else if (i < text.size() && (text[i] == '+' || text[i] == '-')) {
            const int sign = text[i++] == '-' ? -1 : 1;
            int64_t oh, om = 0;
            if (!digits(2, &oh)) return false;
            if (i < text.size() && text[i] == ':') ++i;
            if (i < text.size() && !digits(2, &om)) return false;
            off_s = sign * (oh * 3600 + om * 60);
        }
        if (i != text.size()) return false;
    }
    const int64_t days = days_from_civil(Y, (unsigned)M, (unsigned)D);
    if (unit == 'D') {
        if (has_time) return false;  // (a Date32 cast takes a plain date)
        *out = days;
        return true;
    }
    const int64_t secs = days * 86400 + h * 3600 + mi * 60 + sec - off_s;
    switch (unit) {
        case 's': *out = secs; return true;
        case 'm': *out = secs * 1000 + frac_ns / 1000000; return true;
        case 'u': *out = secs * 1000000 + frac_ns / 1000; return true;
        case 'n': *out = secs * 1000000000 + frac_ns; return true;
    }
    return false;
}

// ---- constant date / timestamp arithmetic: now() / current_timestamp / current_date / today(), DATE / TIMESTAMP literals and
// `+ / - INTERVAL '..'` (README.md:75 of the reference: `created_at > now() - interval '1 day'`). DataFusion folds these at
// planning time (now() is the query's start time); here they fold on the host to a count of nanoseconds since the epoch
// and the comparison is rewritten in the column's own unit. TG_FIXED_NOW_NS pins now() (tests).
struct IntervalMDN {
    int64_t months = 0, days = 0, nanos = 0;
};
// 'N unit [N unit ..]' with unit = year | month | week | day | hour | minute | second | millisecond | microsecond | nanosecond
// (singular / plural, any case); N an integer, or a decimal for the units of a week and below
static bool parse_interval_literal(const std::string& text, IntervalMDN* out) {
    size_t i = 0;
    const size_t n = text.size();
    IntervalMDN iv;
    bool any = false;
    while (true) {
        while (i < n && isspace((unsigned char)text[i])) ++i;
        if (i == n) break;
        size_t j = i;
        if (j < n && (text[j] == '-' || text[j] == '+')) ++j;
        bool digit = false, dot = false;
        while (j < n && (isdigit((unsigned char)text[j]) || (text[j] == '.' && !dot))) {
            if (text[j] == '.') dot = true;
            else digit = true;
            ++j;
        }
        if (!digit) return false;
        const std::string num = text.substr(i, j - i);
        i = j;
        while (i < n && isspace((unsigned char)text[i])) ++i;
        j = i;
        while (j < n && isalpha((unsigned char)text[j])) ++j;
        std::string u = text.substr(i, j - i);
        for (auto& ch : u) ch = (char)tolower((unsigned char)ch);
        if (u.size() > 1 && u.back() == 's') u.pop_back();
        i = j;
        if (u.empty()) u = "second";  // (a bare number counts seconds)
        const double x = atof(num.c_str());
        const long long whole = atoll(num.c_str());
        if (u == "year" || u == "month") {
            if (dot) return false;
            iv.months += whole * (u == "year" ? 12 : 1);
        } else if (u == "week" || u == "day") {
            const double d = x * (u == "week" ? 7.0 : 1.0);
            const double fl = floor(d);
            iv.days += (int64_t)fl;
            iv.nanos += (int64_t)llround((d - fl) * 86400e9);
        } else {
            const double per = u == "hour" ? 3600e9 : u == "minute" ? 60e9 : u == "second" ? 1e9 : u == "millisecond" ? 1e6 : u == "microsecond" ? 1e3
                               : u == "nanosecond" ? 1.0 : 0.0;
            if (per == 0.0) return false;
            iv.nanos += dot ? (int64_t)llround(x * per) : whole * (int64_t)per;
        }
        any = true;
    }
    *out = iv;
    return any;
}
static void civil_from_days(int64_t z, int64_t* y, unsigned* m, unsigned* d) {
    z += 719468;
    const int64_t era = (z >= 0 ? z : z - 146096) / 146097;
    const unsigned doe = (unsigned)(z - era * 146097);
    const unsigned yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
    const unsigned doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
    const unsigned mp = (5 * doy + 2) / 153;
    *d = doy - (153 * mp + 2) / 5 + 1;
    *m = mp < 10 ? mp + 3 : mp - 9;
    *y = (int64_t)yoe + era * 400 + (*m <= 2);
}
constexpr int64_t DAY_NS = 86400ll * 1000000000ll;
static int64_t floor_div(int64_t a, int64_t b) { return a / b - ((a % b != 0) && ((a < 0) != (b < 0))); }
// months first (the day of the month clamped to the target month's length), then days, then the sub-day part
static int64_t add_interval(int64_t ns, const IntervalMDN& iv, int sign) {
    int64_t days = floor_div(ns, DAY_NS);
    const int64_t tod = ns - days * DAY_NS;
    if (iv.months) {
        int64_t y;
        unsigned m, d;
        civil_from_days(days, &y, &m, &d);
        const int64_t mm = y * 12 + (int64_t)(m - 1) + sign * iv.months;
        y = floor_div(mm, 12);
        m = (unsigned)(mm - y * 12) + 1;
        static const unsigned mdays[12] = {31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31};
        const bool leap = (y % 4 == 0 && y % 100 != 0) || y % 400 == 0;
        const unsigned last = m == 2 && leap ? 29 : mdays[m - 1];
        days = days_from_civil(y, m, d < last ? d : last);
    }
    return (days + sign * iv.days) * DAY_NS + tod + sign * iv.nanos;
}
static bool is_fn(const ExprP& x, const char* name, size_t n_args) { return x->kind == Expr::FUNC && x->s == name && x->args.size() == n_args; }
static bool eval_interval(const ExprP& x, IntervalMDN* iv) {
    return is_fn(x, "INTERVAL_LITERAL", 1) && x->args[0]->kind == Expr::LIT_S && parse_interval_literal(x->args[0]->s, iv);
}
// does the tree hold anything only the folding below understands?
static bool has_temporal_fn(const ExprP& x) {
    if (!x) return false;
    if (x->kind == Expr::FUNC && (x->s == "NOW" || x->s == "CURRENT_TIMESTAMP" || x->s == "CURRENT_DATE" || x->s == "TODAY" || x->s == "INTERVAL_LITERAL"))
        return true;
    if (x->kind == Expr::BINARY && (x->s == "+" || x->s == "-")) return has_temporal_fn(x->args[0]) || has_temporal_fn(x->args[1]);
    return false;
}
static bool eval_temporal_const(const ExprP& x, int64_t now_ns, int64_t* ns) {
    if (x->kind == Expr::LIT_S) return parse_temporal_literal(x->s, 'n', ns);
    if ((is_fn(x, "DATE_LITERAL", 1) || is_fn(x, "TIMESTAMP_LITERAL", 1)) && x->args[0]->kind == Expr::LIT_S)
        return parse_temporal_literal(x->args[0]->s, 'n', ns);
    if (is_fn(x, "NOW", 0) || is_fn(x, "CURRENT_TIMESTAMP", 0)) {
        *ns = now_ns;
        return true;
    }
    if (is_fn(x, "CURRENT_DATE", 0) || is_fn(x, "TODAY", 0)) {
        *ns = floor_div(now_ns, DAY_NS) * DAY_NS;
        return true;
    }
    if (x->kind == Expr::BINARY && (x->s == "+" || x->s == "-") && x->args.size() == 2) {
        IntervalMDN iv;
        int64_t base;
        if (eval_temporal_const(x->args[0], now_ns, &base) && eval_interval(x->args[1], &iv)) {
            *ns = add_interval(base, iv, x->s == "+" ? 1 : -1);
            return true;
        }
        if (x->s == "+" && eval_interval(x->args[0], &iv) && eval_temporal_const(x->args[1], now_ns, &base)) {
            *ns = add_interval(base, iv, 1);
            return true;
        }
    }
    return false;
}
static int64_t query_now_ns() {
    if (const char* f = getenv("TG_FIXED_NOW_NS")) return (int64_t)atoll(f);
    timespec ts{};
    clock_gettime(CLOCK_REALTIME, &ts);
    return (int64_t)ts.tv_sec * 1000000000ll + ts.tv_nsec;
}
// `col OP x` for a date / timestamp column and a constant instant x (nanoseconds): the same comparison in the column's unit.
// An x between two ticks of a coarser column (days against a time of day) keeps the comparison exact by moving to the tick
// below: col > x <=> col >= x <=> col > q, col < x <=> col <= x <=> col <= q, col = x never, col <> x always (NULL rows stay NULL).
static ExprP temporal_compare(const ExprP& col_node, const Column& col, const std::string& op_from_col, int64_t x_ns) {
    const int64_t unit = col.temporal_unit == 'D' ? DAY_NS : col.temporal_unit == 's' ? 1000000000ll : col.temporal_unit == 'm' ? 1000000ll
                         : col.temporal_unit == 'u' ? 1000ll : 1ll;
    const int64_t q = floor_div(x_ns, unit);
    const bool exact = q * unit == x_ns;
    auto node = std::make_shared<Expr>();
    node->kind = Expr::BINARY;
    auto lit = std::make_shared<Expr>();
    lit->kind = Expr::LIT_I;
    lit->i = q;
    node->args = {col_node, lit};
    if (exact) node->s = op_from_col;
    else if (op_from_col == ">" || op_from_col == ">=") node->s = ">";
    else if (op_from_col == "<" || op_from_col == "<=") node->s = "<=";
    else {
        node->s = op_from_col == "=" ? "<>" : "=";
        node->args[1] = col_node;
    }
    return node;
}

static ExprP rewrite_string_compares(const ExprP& ex, Engine& e, Table& t, Plan& p, VirtualCols& vc) {
    if (!ex) return ex;
    if (ex->kind == Expr::BINARY && ex->args.size() == 2 && (ex->s == "=" || ex->s == "<>" || ex->s == "<" || ex->s == "<=" || ex->s == ">" || ex->s == ">=")) {
        static const char* const kOps[6] = {"=", "<>", "<", "<=", ">", ">="};
        static const char* const kFlipped[6] = {"=", "<>", ">", ">=", "<", "<="};
        for (int side = 0; side < 2; ++side) {
            const ExprP& c = ex->args[side];
            const ExprP& k = ex->args[1 - side];
            if (c->kind != Expr::COL || !has_temporal_fn(k)) continue;
            Column* col = t.find(c->s);
            if (!col || !col->temporal || !col->temporal_unit) continue;
            int64_t x_ns = 0;
            if (!eval_temporal_const(k, query_now_ns(), &x_ns))
                throw Error(TG_ERR_UNSUPPORTED, "This feature is not implemented: date / timestamp arithmetic beyond <constant> +/- INTERVAL '..'");
            std::string op = ex->s;
            if (side == 1)
                for (int q = 0; q < 6; ++q)
                    if (ex->s == kOps[q]) op = kFlipped[q];
            return temporal_compare(c, *col, op, x_ns);
        }
    }
    // typed literals DATE '..' / TIMESTAMP '..' parse as a function-less pair: the parser hands them over as FUNC nodes
    if (ex->kind == Expr::BINARY && (ex->s == "=" || ex->s == "<>" || ex->s == "<" || ex->s == "<=" || ex->s == ">" || ex->s == ">=")) {
        for (int side = 0; side < 2; ++side) {
            const ExprP& c = ex->args[side];
            ExprP l = ex->args[1 - side];
            if (l->kind == Expr::FUNC && (l->s == "DATE_LITERAL" || l->s == "TIMESTAMP_LITERAL") && l->args.size() == 1) l = l->args[0];
            if (c->kind != Expr::COL || l->kind != Expr::LIT_S) continue;
            Column* col = t.find(c->s);
            if (!col || !col->temporal) continue;
            int64_t v = 0;
            if (!col->temporal_unit || !parse_temporal_literal(l->s, col->temporal_unit, &v))
                throw Error(TG_ERR_INVALID_ARG, "Arrow error: Cast error: Cannot cast string '" + l->s + "' to value of " +
                                                    std::string(col->src_type ? col->src_type : "temporal") + " type");
            auto lit = std::make_shared<Expr>();
            lit->kind = Expr::LIT_I;
            lit->i = v;
            auto copy = std::make_shared<Expr>(*ex);
            copy->args[1 - side] = lit;
            return copy;
        }
    }
    auto utf8_col = [&](const ExprP& x) -> Column* {
        if (!x || x->kind != Expr::COL) return nullptr;
        Column* c = t.find(x->s);
        return c && c->dtype == TG_UTF8 ? c : nullptr;
    };
    // a virtual column of `value_bytes` value bytes followed by `extra` more device bytes (literals, a combined validity)
    auto make_virtual = [&](int32_t dtype, size_t value_bytes, size_t extra, uint8_t** d_extra) -> Column* {
        auto v = std::make_unique<Column>();
        v->name = std::string("\x01str") + std::to_string(vc.cols.size());
        v->dtype = dtype;
        v->n_rows = t.n_rows;
        const size_t bytes = round_up(value_bytes + PAD, PAD), ex_b = round_up(extra + PAD, PAD);
        TG_CUDA(cudaMalloc(&v->values.p, bytes + ex_b));
        TG_CUDA(cudaMemsetAsync(v->values.p, 0, bytes + ex_b, e.stream));
        v->values.cap = bytes + ex_b;
        v->value_bytes = (int64_t)value_bytes;
        *d_extra = v->values.p + bytes;
        vc.cols.push_back(std::move(v));
        return vc.cols.back().get();
    };
    auto col_node = [](const Column* v) {
        auto node = std::make_shared<Expr>();
        node->kind = Expr::COL;
        node->s = v->name;
        return node;
    };
    auto launched = [&]() {
        TG_CUDA(cudaGetLastError());
        e.launches += 1;
        p.stats.launches += 1;
    };
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((t.n_rows + 255) / 256, (int64_t)e.sm_count * 8));
    const size_t words = (size_t)(t.n_rows + 31) / 32;
    static const char* const kCmp[6] = {"=", "<>", "<", "<=", ">", ">="};
    static const int kFlip[6] = {0, 1, 4, 5, 2, 3};  // literal on the left: `'a' < c` is `c > 'a'`
    if (ex->kind == Expr::BINARY) {
        int op = -1;
        for (int k = 0; k < 6; ++k)
            if (ex->s == kCmp[k]) op = k;
        if (op >= 0) {
            Column* ca = utf8_col(ex->args[0]);
            Column* cb = utf8_col(ex->args[1]);
            const ExprP& la = ex->args[0];
            const ExprP& lb = ex->args[1];
            if ((ca && lb->kind == Expr::LIT_S) || (cb && la->kind == Expr::LIT_S)) {
                Column* col = ca ? ca : cb;
                const std::string& lit = ca ? lb->s : la->s;
                if (!ca) op = kFlip[op];
                uint8_t* d_lit = nullptr;
                Column* v = make_virtual(TG_BOOL, words * 4, lit.size() + 1, &d_lit);
                v->validity = col->validity;
                v->validity.owned = false;
                if (!lit.empty()) TG_CUDA(cudaMemcpyAsync(d_lit, lit.data(), lit.size(), cudaMemcpyHostToDevice, e.stream));
                if (t.n_rows > 0) {
                    if (op == 0)  // (equality keeps its own kernel: length test first)
                        str_eq_kernel<<<grid, 256, 0, e.stream>>>((const int32_t*)col->offsets.p, col->values.p, t.n_rows, d_lit, (int32_t)lit.size(),
                                                                  (uint32_t*)v->values.p);
                    else
                        str_cmp_kernel<<<grid, 256, 0, e.stream>>>((const int32_t*)col->offsets.p, col->values.p, nullptr, d_lit, (int32_t)lit.size(), nullptr,
                                                                   nullptr, t.n_rows, op, (uint32_t*)v->values.p, nullptr);
                    launched();
                }
                p.stats.bytes_scanned += (uint64_t)(t.n_rows + 1) * 4 + (uint64_t)col->value_bytes;
                return col_node(v);
            }
            if (ca && cb) {
                uint8_t* d_valid = nullptr;
                const bool any_nulls = ca->validity.p || cb->validity.p;
                Column* v = make_virtual(TG_BOOL, words * 4, any_nulls ? words * 4 : 0, &d_valid);
                if (any_nulls) {
                    v->validity.p = d_valid;
                    v->validity.owned = false;
                    v->null_count = -1;
                }
                if (t.n_rows > 0) {
                    str_cmp_kernel<<<grid, 256, 0, e.stream>>>((const int32_t*)ca->offsets.p, ca->values.p, (const int32_t*)cb->offsets.p, cb->values.p, 0,
                                                               (const uint32_t*)ca->validity.p, (const uint32_t*)cb->validity.p, t.n_rows, op,
                                                               (uint32_t*)v->values.p, any_nulls ? (uint32_t*)d_valid : nullptr);
                    launched();
                }
                p.stats.bytes_scanned += (uint64_t)(t.n_rows + 1) * 8 + (uint64_t)ca->value_bytes + (uint64_t)cb->value_bytes;
                return col_node(v);
            }
        }
    }
    if (ex->kind == Expr::FUNC && ex->args.size() == 1 &&
        (ex->s == "LENGTH" || ex->s == "CHAR_LENGTH" || ex->s == "CHARACTER_LENGTH" || ex->s == "OCTET_LENGTH")) {
        if (Column* col = utf8_col(ex->args[0])) {
            uint8_t* unused = nullptr;
            Column* v = make_virtual(TG_INT64, (size_t)t.n_rows * 8, 0, &unused);
            v->validity = col->validity;
            v->validity.owned = false;
            if (t.n_rows > 0) {
                str_length_kernel<<<grid, 256, 0, e.stream>>>((const int32_t*)col->offsets.p, col->values.p, t.n_rows, ex->s == "OCTET_LENGTH" ? 1 : 0,
                                                              (int64_t*)v->values.p);
                launched();
            }
            p.stats.bytes_scanned += (uint64_t)(t.n_rows + 1) * 4 + (ex->s == "OCTET_LENGTH" ? 0 : (uint64_t)col->value_bytes);
            return col_node(v);
        }
    }
    if (ex->kind == Expr::FUNC && ex->s == "LIKE" && ex->args.size() == 2 && ex->args[1]->kind == Expr::LIT_S) {
        if (Column* col = utf8_col(ex->args[0])) {
            // `%` any sequence, `_` one character, `\` takes the next character literally (DataFusion / arrow-string `like`)
            std::string kind, byte;
            const std::string& pat = ex->args[1]->s;
            for (size_t i = 0; i < pat.size(); ++i) {
                const char ch = pat[i];
                if (ch == '\\' && i + 1 < pat.size()) {
                    kind.push_back(0);
                    byte.push_back(pat[++i]);
                } else if (ch == '%') {
                    if (kind.empty() || kind.back() != 2) {
                        kind.push_back(2);
                        byte.push_back(0);
                    }
                } else if (ch == '_') {
                    kind.push_back(1);
                    byte.push_back(0);
                } else {
                    kind.push_back(0);
                    byte.push_back(ch);
                }
            }
            const size_t m = kind.size();
            uint8_t* d_tok = nullptr;
            Column* v = make_virtual(TG_BOOL, words * 4, 2 * m + 2, &d_tok);
            v->validity = col->validity;
            v->validity.owned = false;
            if (m) {
                TG_CUDA(cudaMemcpyAsync(d_tok, kind.data(), m, cudaMemcpyHostToDevice, e.stream));
                TG_CUDA(cudaMemcpyAsync(d_tok + m, byte.data(), m, cudaMemcpyHostToDevice, e.stream));
                TG_CUDA(cudaStreamSynchronize(e.stream));  // (the token strings are locals)
            }
            if (t.n_rows > 0) {
                str_like_kernel<<<grid, 256, 0, e.stream>>>((const int32_t*)col->offsets.p, col->values.p, t.n_rows, d_tok, d_tok + m, (int32_t)m,
                                                            (uint32_t*)v->values.p);
                launched();
            }
            p.stats.bytes_scanned += (uint64_t)(t.n_rows + 1) * 4 + (uint64_t)col->value_bytes;
            return col_node(v);
        }
    }
    auto copy = std::make_shared<Expr>(*ex);
    for (auto& a : copy->args) a = rewrite_string_compares(a, e, t, p, vc);
    return copy;
}

void exec_scan_jobs(Engine& e, Table& t, Plan& p, const std::vector<int>& agg_ids) {
    VirtualCols virtuals(e);
    std::vector<ScanOp> ops;
    uint64_t bytes = 0;
    std::vector<Column*> counted_vals, counted_bits;
    auto count_bytes = [&](Column* c, bool values) {
        if (values && std::find(counted_vals.begin(), counted_vals.end(), c) == counted_vals.end()) {
            counted_vals.push_back(c);
            bytes += c->dtype == TG_BOOL ? (uint64_t)(t.n_rows + 7) / 8 : (uint64_t)t.n_rows * 8;
        }
        if (c->validity.p && std::find(counted_bits.begin(), counted_bits.end(), c) == counted_bits.end()) {
            counted_bits.push_back(c);
            bytes += (uint64_t)(t.n_rows + 7) / 8;
        }
    };
    // COUNT(c) of a column that also has a NUM aggregate in this plan comes for free from that unit's n
    std::vector<std::pair<int, int>> valid_from_num;  // (valid agg, num agg)
    for (int id : agg_ids) {
        Agg& a = p.aggs[id];
        if (a.err != TG_OK) continue;
        if (a.kind == A_VALID) {
            bool folded = false;
            for (int id2 : agg_ids) {
                const Agg& b = p.aggs[id2];
                Column* bc = b.kind == A_NUM && b.err == TG_OK ? t.find(b.cols[0]) : nullptr;
                if (bc && b.cols[0] == a.cols[0] && (bc->dtype == TG_INT64 || bc->dtype == TG_FLOAT64) && bc->validity.p) {
                    valid_from_num.emplace_back(id, id2);
                    folded = true;
                    break;
                }
            }
            if (folded) continue;
        }
        ScanOp o;
        o.agg = id;
        auto col = [&](const std::string& name) -> Column* {
            Column* c = t.find(name);
            if (!c) {
                a.err = TG_ERR_COLUMN_NOT_FOUND;
                a.err_msg = no_field_msg(t, name);
            }
            return c;
        };
        auto numeric = [&](Column*& c) {  // (Int32 / Float32: replaced by the widened shadow)
            if (Column* v = c->temporal ? nullptr : numeric_view(e, c)) {
                if (v != c || c->src_type) {
                    a.narrow = 1 | (c->src_unsigned ? 2 : 0);
                    a.narrow_name = c->src_type ? c->src_type : (c->dtype == TG_INT32 ? "Int32" : "Float32");
                }
                c = v;
                return true;
            }
            a.err = TG_ERR_TYPE_MISMATCH;
            a.err_msg = "Error during planning: numeric aggregate is not supported for column '" + c->name +
                        "' of this type";
            return false;
        };
        switch (a.kind) {
            case A_VALID: {
                Column* c = col(a.cols[0]);
                if (!c) break;
                if (!c->validity.p) {  // no nulls: COUNT(c) == COUNT(*) without touching the device
                    a.u[0] = (uint64_t)t.n_rows;
                    a.u[1] = (uint64_t)t.n_rows;
                    break;
                }
                o.kind = UNIT_COUNT;
                o.c0 = c;
                o.cost = 0.2;
                count_bytes(c, false);
                ops.push_back(std::move(o));
            } break;
            case A_NUM: {
                Column* c = col(a.cols[0]);
                if (!c || !numeric(c)) break;
                o.kind = c->dtype == TG_INT64 ? UNIT_NUM_I64 : UNIT_NUM_F64;
                o.c0 = c;
                o.flags = a.flags ? a.flags : 7;
                if (c->dtype != TG_INT64) o.flags &= ~4;
                // warp-instructions per 32 rows: load + mask, then moments / min-max / integer sum
                // warp-instructions per 32 rows of the specialised loops (counted in the SASS)
                o.cost = 2.5 + ((o.flags & 1) ? 5.5 : 0.0) + ((o.flags & 2) ? (c->dtype == TG_INT64 ? 8.5 : 6.5) : 0.0) +
                         ((o.flags & 4) ? 3.5 : 0.0) + ((o.flags & 1) && c->dtype == TG_INT64 ? 1.0 : 0.0);
                count_bytes(c, true);
                ops.push_back(std::move(o));
            } break;
            case A_PAIR: {
                Column* x = col(a.cols[0]);
                if (!x) break;
                Column* y = col(a.cols[1]);
                if (!y || !numeric(x) || !numeric(y)) break;
                o.kind = UNIT_PAIR;
                o.c0 = x;
                o.c1 = y;
                o.cost = 15.5 + (x->dtype == TG_INT64 ? 1.0 : 0.0) + (y->dtype == TG_INT64 ? 1.0 : 0.0);
                count_bytes(x, true);
                count_bytes(y, true);
                ops.push_back(std::move(o));
            } break;
            case A_PRED: {
                if (!a.expr) break;
                try {
                    const ExprP expr = rewrite_string_compares(a.expr, e, t, p, virtuals);
                    ColumnResolver res = [&](const std::string& name) -> ColumnBinding {
                        Column* c = t.find(name);
                        if (!c && !name.empty() && name[0] == '\x01')
                            for (auto& v : virtuals.cols)
                                if (v->name == name) c = v.get();
                        if (!c) throw Error(TG_ERR_COLUMN_NOT_FOUND, no_field_msg(t, name));
                        if (c->dtype == TG_INT32 || c->dtype == TG_FLOAT32) c = numeric_view(e, c);
                        for (size_t i = 0; i < o.pred_cols.size(); ++i)
                            if (o.pred_cols[i] == c) return ColumnBinding{(int)i, c->dtype};
                        o.pred_cols.push_back(c);
                        return ColumnBinding{(int)o.pred_cols.size() - 1, c->dtype};
                    };
                    bool is_or = false;
                    if (try_compile_terms(expr, res, o.terms, is_or)) {
                        o.kind = UNIT_TERMS;
                        o.flags = is_or ? 1 : 0;
                        o.cost = 1.0 + 6.5 * (double)o.terms.size();
                    } else {
                        o.pred_cols.clear();
                        compile_predicate(expr, res, o.code);
                        o.kind = UNIT_PRED;
                        o.cost = 10.0 + 25.0 * (double)o.code.size();
                    }
                } catch (Error& er) {
                    a.err = er.code;
                    a.err_msg = er.msg;
                    break;
                }
                for (auto* c : o.pred_cols) count_bytes(c, true);
                ops.push_back(std::move(o));
            } break;
            default: break;
        }
    }
    p.stats.bytes_scanned += bytes;
    struct FoldFill {
        Plan& p;
        Table& t;
        std::vector<std::pair<int, int>>& v;
        ~FoldFill() {
            if (p_fused) {  // the NUM aggregate's count only exists on the device: scan_payload_kernel folds it
                for (auto& pr : v) p_fused->folds.push_back(pr);
                return;
            }
            for (auto& pr : v) {
                p.aggs[pr.first].u[0] = (uint64_t)t.n_rows;
                p.aggs[pr.first].u[1] = p.aggs[pr.second].u[0];
            }
        }
        FusedScan* p_fused;
    } fold_fill{p, t, valid_from_num, e.fused};
    if (t.n_rows == 0) {
        // nothing to scan: aggregates keep their zero state (COUNT(*) = 0)
        for (auto& o : ops)
            if (p.aggs[o.agg].kind == A_PRED) p.aggs[o.agg].u[2] = 0;
        return;
    }
    // Split into passes. A pass of at most SCAN_CONSUMER_WARPS aggregates gives every consumer warp ONE unit whose
    // state stays in registers; beyond that the kernel keeps per-lane state in shared memory and runs ~3x slower
    // (measured: 80 % -> 26 % of the HBM peak on the full numeric set), so re-reading a column in a second fast pass
    // is the better deal. Aggregates are ordered by their first column so a column's aggregates share a pass.
    // (by the column's ORDINAL in the table, never its address: the unit layout — and with it the order of the
    // floating-point sums — must not depend on where the heap put the Column objects)
    auto ordinal = [&](const ScanOp& o) {
        const Column* c = o.c0 ? o.c0 : (o.pred_cols.empty() ? nullptr : o.pred_cols[0]);
        if (!c) return -1;
        for (size_t i = 0; i < t.cols.size(); ++i)
            if (t.cols[i].get() == c || t.cols[i]->wide.get() == c) return (int)i;
        return (int)t.cols.size();
    };
    std::vector<std::pair<int, size_t>> op_key(ops.size());
    for (size_t i = 0; i < ops.size(); ++i) op_key[i] = {ordinal(ops[i]), i};
    std::stable_sort(op_key.begin(), op_key.end(), [](const std::pair<int, size_t>& a, const std::pair<int, size_t>& b) { return a.first < b.first; });
    {
        std::vector<ScanOp> sorted;
        sorted.reserve(ops.size());
        for (auto& k : op_key) sorted.push_back(std::move(ops[k.second]));
        ops.swap(sorted);
    }
    // A pass is also bounded by the kernel's tables: SCAN_MAX_TERMS predicate terms, SCAN_MAX_COLS tile columns and
    // SCAN_MAX_CODE predicate instructions. The reference evaluates every constraint on its own, so a suite never fails
    // as a whole: a pass is closed before an op would overflow a table, and an op that cannot fit even alone fails
    // only its own aggregate.
    auto op_cols = [](const ScanOp& o, std::vector<const Column*>& out) {
        auto add = [&](const Column* c) {
            if (c && std::find(out.begin(), out.end(), c) == out.end()) out.push_back(c);
        };
        add(o.c0);
        add(o.c1);
        for (auto* c : o.pred_cols) add(c);
    };
    size_t i = 0;
    while (i < ops.size()) {
        std::vector<ScanOp> pass;
        int code = 0, terms = 0;
        std::vector<const Column*> cols;
        while (i < ops.size() && pass.size() < (size_t)SCAN_CONSUMER_WARPS) {
            const int add_code = (int)ops[i].code.size();
            const int add_terms = ops[i].kind == UNIT_TERMS ? (int)ops[i].terms.size() : 0;
            std::vector<const Column*> with = cols;
            op_cols(ops[i], with);
            if (!pass.empty() && (code + add_code > SCAN_MAX_CODE || terms + add_terms > SCAN_MAX_TERMS || with.size() > (size_t)SCAN_MAX_COLS)) break;
            code += add_code;
            terms += add_terms;
            cols.swap(with);
            pass.push_back(std::move(ops[i]));
            ++i;
        }
        std::vector<int> pass_aggs;
        for (auto& o : pass) pass_aggs.push_back(o.agg);
        try {
            run_scan_pass(e, t, p, pass);
        } catch (Error& er) {
            if (er.code == TG_ERR_CUDA) throw;
            for (int id : pass_aggs) {
                p.aggs[id].err = er.code;
                p.aggs[id].err_msg = er.msg;
            }
        }
    }
}

// ------------------------------------------------------------------ execute ----

void execute_partial(Engine& e, Plan& p, const std::string& table_name) {
    std::lock_guard<std::mutex> g(e.mu);
    TG_CUDA(cudaSetDevice(e.device));
    p.reset_partials();
    p.stats = tg_exec_stats{};
    p.executed = false;
    e.sync_copies();
    auto it = e.tables.find(table_name);
    Table* t = it == e.tables.end() ? nullptr : it->second.get();
    std::vector<int> scan_ids, string_ids, kll_ids, length_ids, grouped_ids;
    for (size_t i = 0; i < p.aggs.size(); ++i) {
        Agg& a = p.aggs[i];
        if (a.err != TG_OK) continue;
        if (a.kind == A_FK) continue;  // uses its own tables
        if ((a.kind == A_DISTINCT || a.kind == A_SPEARMAN) && !a.redirect[0].empty()) continue;  // reads the shuffled / gathered table instead
        if (!t) {
            a.err = TG_ERR_TABLE_NOT_FOUND;
            a.err_msg = "Error during planning: table 'datafusion.public." + table_name + "' not found";
            continue;
        }
        switch (a.kind) {
            case A_ROWS:
                a.u[0] = (uint64_t)t->n_rows;
                a.u[1] = (uint64_t)t->cols.size();  // schema width (ColumnCountConstraint)
                break;
            case A_VALID:
            case A_NUM:
            case A_PAIR:
            case A_PRED: scan_ids.push_back((int)i); break;
            case A_REGEX: string_ids.push_back((int)i); break;
            case A_KLL: kll_ids.push_back((int)i); break;
            case A_LENGTH: length_ids.push_back((int)i); break;
            case A_GROUPED: grouped_ids.push_back((int)i); break;
            default: break;
        }
    }
    if (t && !scan_ids.empty()) exec_scan_jobs(e, *t, p, scan_ids);
    if (t && !string_ids.empty()) exec_string_jobs(e, *t, p, string_ids);
    if (t && !length_ids.empty()) exec_length_jobs(e, *t, p, length_ids);
    if (t && !kll_ids.empty()) exec_kll_jobs(e, *t, p, kll_ids);
    if (t && !grouped_ids.empty()) exec_grouped_jobs(e, *t, p, grouped_ids);
    for (size_t i = 0; i < p.aggs.size(); ++i) {
        Agg& a = p.aggs[i];
        if (a.err != TG_OK) continue;
        try {
            switch (a.kind) {
                case A_DISTINCT:
                case A_SPEARMAN: {
                    Table* dt = t;
                    if (!a.redirect[0].empty()) {
                        auto rit = e.tables.find(a.redirect[0]);
                        if (rit == e.tables.end())
                            throw Error(TG_ERR_TABLE_NOT_FOUND, "Error during planning: table 'datafusion.public." + a.redirect[0] + "' not found");
                        dt = rit->second.get();
                    }
                    if (a.kind == A_DISTINCT) exec_distinct_job(e, *dt, p, (int)i);
                    else exec_spearman_job(e, *dt, p, (int)i);
                } break;
                case A_FK: exec_fk_job(e, p, (int)i); break;
                case A_HIST: exec_hist_job(e, *t, p, (int)i); break;
                default: break;
            }
        } catch (Error& er) {
            if (er.code == TG_ERR_CUDA) throw;
            a.err = er.code;
            a.err_msg = er.msg;
        }
    }
}

// ------------------------------------------------------------------ fused multi-GPU step (scan-only plans) ----
bool execute_exchange_fused(Engine& e, Plan& p, const std::string& table_name) {
    std::unique_lock<std::mutex> g(e.mu);
    TG_CUDA(cudaSetDevice(e.device));
    Mailbox& m = e.mailbox;
    if (!m.open) return false;
    const int n_aggs = (int)p.aggs.size();
    // rank-independent decisions only: the plan is the same on every rank
    for (auto& a : p.aggs)
        if (a.kind != A_ROWS && a.kind != A_VALID && a.kind != A_NUM && a.kind != A_PAIR && a.kind != A_PRED) return false;
    const size_t payload = 16 + (size_t)n_aggs * sizeof(DevAggRec);
    const size_t pinned_need = (size_t)n_aggs * (sizeof(DevAggRec) + sizeof(ScanOpMeta) + 1 + sizeof(int2)) + 256;
    if (n_aggs == 0 || payload > m.slot_bytes || pinned_need > m.slot_bytes) return false;

    p.reset_partials();
    p.stats = tg_exec_stats{};
    p.executed = false;
    e.sync_copies();
    auto it = e.tables.find(table_name);
    Table* t = it == e.tables.end() ? nullptr : it->second.get();
    // device block: states | metas | template | from_device | folds   (the payload itself is assembled in the mailbox's d_stage)
    const size_t st_b = round_up((size_t)n_aggs * sizeof(DevAggRec), 256), me_b = round_up((size_t)n_aggs * sizeof(ScanOpMeta), 256);
    const size_t fd_b = round_up((size_t)n_aggs, 256), fo_b = round_up((size_t)n_aggs * sizeof(int2), 256);
    uint8_t* d = e.aux(2 * st_b + me_b + fd_b + fo_b + 256);
    FusedScan fz;
    fz.d_states = (DevAggRec*)d;
    fz.d_metas = (ScanOpMeta*)(d + st_b);
    DevAggRec* d_tmpl = (DevAggRec*)(d + st_b + me_b);
    uint8_t* d_from = d + 2 * st_b + me_b;
    int2* d_folds = (int2*)(d + 2 * st_b + me_b + fd_b);
    // pinned staging: the mailbox's host stage (unused by this path otherwise)
    uint8_t* hp = m.h_stage;
    fz.h_metas = (ScanOpMeta*)hp;
    DevAggRec* h_tmpl = (DevAggRec*)(hp + me_b);
    uint8_t* h_from = hp + me_b + st_b;
    int2* h_folds = (int2*)(hp + me_b + st_b + fd_b);
    if (me_b + st_b + fd_b + fo_b > m.slot_bytes) return false;
    fz.from_device.assign((size_t)n_aggs, 0);
    TG_CUDA(cudaMemsetAsync(fz.d_states, 0, st_b, e.stream));

    std::vector<int> scan_ids;
    for (int i = 0; i < n_aggs; ++i) {
        Agg& a = p.aggs[i];
        if (a.err != TG_OK) continue;
        if (!t) {
            a.err = TG_ERR_TABLE_NOT_FOUND;
            a.err_msg = "Error during planning: table 'datafusion.public." + table_name + "' not found";
            continue;
        }
        if (a.kind == A_ROWS) {
            a.u[0] = (uint64_t)t->n_rows;
            a.u[1] = (uint64_t)t->cols.size();
        } else {
            scan_ids.push_back(i);
        }
    }
    struct Unfuse {
        Engine& e;
        ~Unfuse() { e.fused = nullptr; }
    } unfuse{e};
    e.fused = &fz;
    if (t && !scan_ids.empty()) exec_scan_jobs(e, *t, p, scan_ids);
    e.fused = nullptr;
    // the template: everything the host knows (kinds, error codes, host-resolved states)
    for (int i = 0; i < n_aggs; ++i) {
        const Agg& a = p.aggs[i];
        DevAggRec r{};
        r.kind = (uint64_t)a.kind;
        r.err = (uint64_t)a.err;
        memcpy(r.u, a.u, 64);
        memcpy(r.f, a.f, 64);
        h_tmpl[i] = r;
        h_from[i] = a.err == TG_OK ? fz.from_device[i] : 0;
    }
    const int n_folds = (int)fz.folds.size();
    for (int i = 0; i < n_folds; ++i) h_folds[i] = make_int2(fz.folds[i].first, fz.folds[i].second);
    // template / flags / folds are read from pinned host memory by the kernel itself (a few hundred bytes over PCIe inside
    // the kernel cost less than three copy calls on the stream)
    (void)d_tmpl;
    (void)d_from;
    (void)d_folds;
    scan_payload_kernel<<<1, 128, 0, e.stream>>>(h_tmpl, h_from, fz.d_states, h_folds, n_folds, n_aggs, t ? (uint64_t)t->n_rows : 0ull, m.d_stage);
    TG_CUDA(cudaGetLastError());
    e.launches += 1;
    p.stats.launches += 1;
    std::vector<std::vector<uint8_t>> all;
    mailbox_exchange_device(e, payload, all);  // publish + collect + the step's one synchronisation
    float ms = 0;
    if (t && !scan_ids.empty() && cudaEventElapsedTime(&ms, e.ev[0], e.ev[1]) == cudaSuccess) {  // the (last) scan pass
        p.stats.scan_ms += ms;
        p.stats.gpu_ms += ms;
    } else {
        cudaGetLastError();
    }
    // rank-ordered merge (deterministic), then finalize
    std::vector<std::pair<tg_status, std::string>> local_err;
    for (auto& a : p.aggs) local_err.emplace_back(a.err, a.err_msg);
    p.reset_partials();
    static const std::vector<uint8_t> no_blob;
    for (int r = 0; r < m.world; ++r) {
        const std::vector<uint8_t>& b = all[r];
        uint64_t na = 0;
        if (b.size() >= 8) memcpy(&na, b.data(), 8);
        if (na != (uint64_t)n_aggs || b.size() < 8 + (size_t)n_aggs * sizeof(DevAggRec))
            throw Error(TG_ERR_INVALID_ARG, "fused exchange: rank " + std::to_string(r) + " published the states of another plan");
        for (int i = 0; i < n_aggs; ++i) {
            DevAggRec rec;
            memcpy(&rec, b.data() + 8 + (size_t)i * sizeof(DevAggRec), sizeof(rec));
            if ((int32_t)rec.kind != p.aggs[i].kind) throw Error(TG_ERR_INVALID_ARG, "fused exchange: aggregate kinds differ between ranks");
            const tg_status err = (tg_status)rec.err;
            const std::string msg = err == TG_OK ? std::string()
                                   : (r == m.rank || local_err[i].first == err) && !local_err[i].second.empty()
                                       ? local_err[i].second
                                       : "error " + std::to_string((int)err) + " on rank " + std::to_string(r);
            p.merge_state(i, err, msg, rec.u, rec.f, no_blob);
        }
    }
    g.unlock();
    p.finalize();
    return true;
}

}  // namespace tg
