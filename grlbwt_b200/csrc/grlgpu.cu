// C ABI (include/grlgpu.h) and host-side sequencing of one parse round on one B200.
// Replaces the strategy + par_round pair of the reference (lib/exact_algo/exact_par_phase.cpp:265-497).
#include "../../include/grlgpu.h"
#include "util.cuh"
#include "primitives.cuh"
#include "parse_kernels.cuh"
#include "dict_kernels.cuh"
#include "comm.hpp"

#include <algorithm>
#include <cstring>
#include <memory>
#include <vector>

using namespace grl;


// the artefacts of one level on the device: tot rules (rule_l / rule_r of sym_bytes each, has_hocc) and n_pre preliminary-BWT runs
struct DevLevel {
    int sym_bytes = 4;
    u64 tot = 0, n_pre = 0;
    DevBuf<u8> rule_l, rule_r, has_hocc, pre_sym;
    DevBuf<u64> pre_len;
    bool present() const { return rule_l.p != nullptr; }
};

// the level one call acts on (not owning): the last round's level, this rank's slice of a multi-GPU level, or a kept level
struct LevelView {
    int sym_bytes;
    u64 tot, n_pre, rank_base;  // rank_base: global rank of the first rule (checksum weights)
    const void *rule_l, *rule_r;
    const u8* has_hocc;
    const void* pre_sym;
    const u64* pre_len;
};
// pre_drop: leading runs of the arrays that belong to another rank
inline LevelView view_of(const DevLevel& L, u64 rank_base = 0, u64 pre_drop = 0) {
    return {L.sym_bytes, L.tot, L.n_pre - pre_drop, rank_base, L.rule_l.p, L.rule_r.p, L.has_hocc.p, L.pre_sym.p + pre_drop * (u64)L.sym_bytes, L.pre_len.p + pre_drop};
}

// level slice of the last multi-GPU round (owned by the context until the next round / fetch): lvl.tot rules from global rank
// rank_base on; runs [pre_drop, lvl.n_pre) of lvl.pre_* are this rank's and go to global run pre_first on
struct Mg2Slices {
    DevLevel lvl;
    u64 rank_base = 0, tot_global = 0;
    u64 pre_drop = 0, pre_first = 0, n_pre_global = 0;
    bool valid = false;
    LevelView view() const { return view_of(lvl, rank_base, pre_drop); }
};

// device-side induction (induce.cuh): a level's BWT as maximal runs, and a level kept on the device for it
struct IndBwt {
    DevBuf<u32> sym, len;
    u32 n_runs = 0, n_syms = 0;
};

struct IndLevel {  // a kept level (device): 32-bit symbols
    u64 alphabet = 0;
    DevLevel lvl;
};

// a level handed over until grlgpu_fetch_wait: its arrays, and the 32-bit run lengths when the host takes those
struct ParkedLevel {
    DevLevel lvl;
    DevBuf<u32> len32;
};

// the LF table of a .rl_bwt image (invert.cuh, part a): runs, run starts, F rows, E[j] = {LF(j) << 32 | BWT[j]}
struct LfTable {
    u64 n = 0, n_runs = 0, N = 0;   // BWT length, records, separators
    u32 sep = 0;                    // smallest symbol of a non-empty record
    DevBuf<u32> sym, len, start, F; // start has n_runs + 1 entries
    DevBuf<u32> order;              // run indices in (symbol, run index) order
    DevBuf<u64> E;
};

// a loaded FM-index (fm.cuh): the LF table, a symbol directory, psi, and the locate table and extract samples once some call needed them
struct FmIndex {
    LfTable t;
    u64 n_dir = 0;
    DevBuf<u32> dir_sym, dir_first, dir_C;  // per distinct symbol: the symbol, its slice [dir_first[d], dir_first[d + 1]) of t.order, C[c]
    DevBuf<u32> psi;                        // psi[LF(j)] = j
    DevBuf<u64> doc;                        // locate table: {string << 32 | offset} for every row
    bool doc_ready = false;
    DevBuf<u32> samp, samp_off;             // extract samples: the row at offset s * FM_EXTRACT_SAMPLE of string k is samp[samp_off[k] + s]
    bool samp_ready = false;
};

struct grlgpu_ctx {
    int device = 0;
    int n_sm = 148;
    u64 flags = 0;
    cudaStream_t st = nullptr;
    bool own_stream = true;
    std::string last_error;
    DevicePool pool;  // declared before every DevBuf member: destroyed after them
    Profiler prof;

    // current text
    const void* text = nullptr;  // device
    DevBuf<u8> text_own;         // owns `text` unless borrowed
    u64 n = 0;
    int w = 0;
    bool first = true;
    DevBuf<u32> end_bits;   // string-end bitmap of the current text (rounds >= 2)
    DevBuf<u8> is_suffix;   // per symbol of the current alphabet (rounds >= 2)
    u64 alphabet = 0;       // A
    u64 n_strings = 0;
    u64 sep = 0;
    int round = 0;
    bool done = false;
    bool have_stats = false;
    grlgpu_stats_t stats{};
    u64 hist[256] = {0};  // byte alphabets: histogram of the (local) text

    // artefacts of the last round (device)
    DevLevel lvl;
    u64 lvl_alphabet = 0;
    u64 lvl_n_in = ~0ull;  // upper bound of the sum of the level's run lengths (all ones: unknown)

    // asynchronous level fetches: a second stream copies while the next round computes; the level's device buffers
    // are parked here (not returned to the pool) until grlgpu_fetch_wait
    cudaStream_t copy_st = nullptr;
    cudaEvent_t copy_ev = nullptr;
    std::vector<ParkedLevel> parked;

    // streaming ingest (grlgpu_text_begin / _stage / _commit / _end): two pinned staging buffers, H2D on the copy stream
    u8* stage_buf[2] = {nullptr, nullptr};
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};
    u64 stage_cap = 0, ingest_off = 0, ingest_bytes = 0;
    int stage_cur = 0;
    bool ingesting = false;

    // device-side induction: levels kept on the device (grlgpu_keep_level / grlgpu_level_adopt) and the resulting level-0 BWT
    std::vector<IndLevel> kept;
    IndBwt bwt_dev;
    bool bwt_ready = false;

    // multi-GPU rounds (mg2.cuh): global string count, this rank's slices of the last level, bytes it sent in the last round
    u64 mg_n_strings = 0;
    Mg2Slices mg_sl;
    u64 mg_exchange_bytes = 0, mg_parse_len_local = 0, mg_n_in_local = 0;

    // optional: dictionary of the last round kept for tests (GRLGPU_FLAG_KEEP_DICT)
    u64 kd_d = 0, kd_nE = 0, kd_nS = 0;
    DevBuf<u8> kd_D;
    DevBuf<u32> kd_off, kd_len, kd_order, kd_phr_of;
    DevBuf<u64> kd_freq, kd_meta;

    // FM-index of a .rl_bwt image (grlgpu_fm_load), at most one
    std::unique_ptr<FmIndex> fm;
};

namespace {

struct Timer {
    cudaEvent_t a{}, b{};
    cudaStream_t st;
    explicit Timer(cudaStream_t s) : st(s) {
        GRL_CUDA(cudaEventCreate(&a));
        GRL_CUDA(cudaEventCreate(&b));
    }
    ~Timer() { cudaEventDestroy(a); cudaEventDestroy(b); }
    void start() { GRL_CUDA(cudaEventRecord(a, st)); }
    void stop() { GRL_CUDA(cudaEventRecord(b, st)); }
    float ms() {
        GRL_CUDA(cudaEventSynchronize(b));
        float t = 0;
        GRL_CUDA(cudaEventElapsedTime(&t, a, b));
        return t;
    }
};

template <class T>
T d2h_scalar(const T* dptr, cudaStream_t st) {
    static_assert(sizeof(T) % 4 == 0, "d2h_scalar reads whole words");
    T h;
    d2h_small(&h, dptr, sizeof(T), st);
    return h;
}

inline unsigned grid_for(u64 n, int threads) { return (unsigned)std::max<u64>(1, div_up(n, (u64)threads)); }

static __global__ void table_init_kernel(ulonglong2* table, u64 cap) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cap) table[i] = make_ulonglong2(HT_EMPTY, 0ULL);
}
static __global__ void next_start_bits_kernel(const u32* __restrict__ end_bits, u64 n, u32* __restrict__ start_bits) {
    // start_bits[q] = (q == 0) || end_bits[q-1]   (string starts of the current text)
    const u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 n_words = (n + 31) / 32;
    if (w >= n_words) return;
    u32 cur = end_bits[w];
    u32 prev = w ? end_bits[w - 1] : 0x80000000u;
    u32 s = (cur << 1) | (prev >> 31);
    if (w == n_words - 1 && (n & 31)) s &= (1u << (n & 31)) - 1u;
    start_bits[w] = s;
}
template <class CellT>
__global__ void __launch_bounds__(256) first_round_end_bits_kernel(const CellT* __restrict__ text, u64 n, CellT sep, u32* __restrict__ end_bits) {
    // thread = 32 cells = one bitmap word, 16-byte vector loads
    const u64 word = (u64)blockIdx.x * blockDim.x + threadIdx.x, base = word * 32;
    if (base >= n) return;
    const u64 cnt = n - base;
    u32 bits = 0;
    if (cnt >= 32) {
        __align__(16) CellT c[32];
        constexpr int NV = 32 * sizeof(CellT) / 16;
        const uint4* src = reinterpret_cast<const uint4*>(text + base);
        uint4* dst = reinterpret_cast<uint4*>(c);
#pragma unroll
        for (int k = 0; k < NV; k++) dst[k] = src[k];
#pragma unroll
        for (int k = 0; k < 32; k++) bits |= (u32)(c[k] == sep) << k;
    } else {
        for (u64 k = 0; k < cnt; k++) bits |= (u32)(text[base + k] == sep) << k;
    }
    end_bits[word] = bits;
}
static __global__ void adjacent_max_diff_kernel(const u64* __restrict__ ptrs, u64 n_str, u64* out) {
    u64 m = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_str; i += (u64)gridDim.x * blockDim.x) {
        const u64 dlt = ptrs[i + 1] - ptrs[i];
        m = dlt > m ? dlt : m;
    }
    m = warp_max(m);
    if (lane_id() == 0 && m) atomicMax(out, m);
}
static __global__ void u32_to_u64_kernel(const u32* __restrict__ in, u64 n, u64* __restrict__ out) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i];
}

// state shared by the stages of one round
struct Round {
    grlgpu_ctx* c;
    cudaStream_t st;
    u64 n, p = 0, d = 0, nE = 0, cap = 0, G = 0, tot = 0, n_pre = 0, max_freq = 0, max_len = 0;
    DevBuf<u32> start_bits, end_bits_first;
    const u32* end_bits = nullptr;  // of the input text
    DevBuf<ulonglong2> table;
    DevBuf<u32> slot_of_phrase, occ_slots;
    DevBuf<u64> ph_pos, ph_freq;
    DevBuf<u32> ph_len, ph_off;
    DevBuf<u8> D_raw;
    DevBuf<u32> phr_of, rem, rank, order;
    DevBuf<ulonglong2> einfo;
    // suffix-order plan: K symbol codes of sym_bits bits per 64-bit key; ext_mode = refinement by key extension, over the
    // nS valid entries only (first keys + entry ids come out of the dictionary gather); else prefix doubling over all nE
    int sym_bits = 0, K = 1, spare = 0;  // spare: bits of the first key beyond the K whole codes (key extension only)
    bool ext_mode = false;
    u64 nS = 0;
    DevBuf<u64> keys;
    DevBuf<u32> vals;
    const void* dict_text = nullptr;  // multi-GPU partition: the received phrase cells its ph_pos point into
    explicit Round(grlgpu_ctx* ctx) : c(ctx), st(ctx->st), n(ctx->n) {}
};

// ---------------- text stage: boundary flags -> phrase starts -> dedup table -> distinct list ----------------
template <class CellT, bool FIRST>
void stage_flags(Round& R) {
    grlgpu_ctx* c = R.c;
    const CellT* text = (const CellT*)c->text;
    const u64 n_words = div_up(R.n, 32);
    const u64 n_blocks = div_up(n_words, LMS_THREADS);
    R.start_bits.alloc(n_words, R.st);
    u32* end_out = nullptr;
    if (FIRST) {
        R.end_bits_first.alloc(n_words, R.st);
        end_out = R.end_bits_first.p;
        R.end_bits = R.end_bits_first.p;
    } else R.end_bits = c->end_bits.p;
    const u32* end_in = FIRST ? nullptr : c->end_bits.p;
    DevBuf<u32> need_slow(1, R.st);
    need_slow.zero();
    const CellT sep = (CellT)c->sep;
    bool slow = (c->flags & GRLGPU_FLAG_FORCE_SLOW_SCAN) != 0;
    if (!slow) {
        GRL_LAUNCH("lms_flags", R.n * sizeof(CellT) + R.n / 4, (lms_flags_kernel<CellT, FIRST, 0>), (unsigned)n_blocks, LMS_THREADS, 0, R.st, text, R.n, sep, end_in, end_out, R.start_bits.p, nullptr, nullptr, need_slow.p);
        slow = d2h_scalar(need_slow.p, R.st) != 0;
    }
    if (slow) {  // a run of equal cells crosses a CTA boundary by more than the look-ahead
        DevBuf<u8> state(n_blocks, R.st), incoming(n_blocks, R.st);
        GRL_LAUNCH("lms_flags", R.n * sizeof(CellT) + R.n / 4, (lms_flags_kernel<CellT, FIRST, 1>), (unsigned)n_blocks, LMS_THREADS, 0, R.st, text, R.n, sep, end_in, end_out, R.start_bits.p, state.p, nullptr, need_slow.p);
        GRL_LAUNCH("lms_resolve", 0, lms_resolve_kernel, 1, 32, 0, R.st, state.p, incoming.p, n_blocks);
        GRL_LAUNCH("lms_flags", R.n * sizeof(CellT) + R.n / 4, (lms_flags_kernel<CellT, FIRST, 2>), (unsigned)n_blocks, LMS_THREADS, 0, R.st, text, R.n, sep, end_in, end_out, R.start_bits.p, nullptr, incoming.p, need_slow.p);
        GRL_CUDA(cudaStreamSynchronize(R.st));
    }
}

void dict_offsets(Round& R);

template <class CellT, class PosT>
void insert_uncached(Round& R, BitmapCompactor& bc, DevBuf<u8>& ps_raw, u64 j0, u64 cap, u32* overflow) {
    grlgpu_ctx* c = R.c;
    if (!ps_raw.p) {  // compacted phrase starts (top bit: starts a string), sentinel ps[p] = n | FLAG
        ps_raw.alloc((R.p + 1) * sizeof(PosT), R.st);
        bc.write<PosT>(R.end_bits, (PosT*)ps_raw.p);
        const PosT sentinel = (PosT)R.n | PosFlag<PosT>::FLAG;
        GRL_CUDA(cudaMemcpyAsync((PosT*)ps_raw.p + R.p, &sentinel, sizeof(PosT), cudaMemcpyHostToDevice, R.st));
        GRL_CUDA(cudaStreamSynchronize(R.st));
    }
    const u64 cnt = R.p - j0;
    GRL_LAUNCH("phrase_insert", (R.n + cnt) * sizeof(CellT) + cnt * (2 * sizeof(PosT) + 4 + 32), (phrase_insert_kernel<CellT, PosT>), grid_for(cnt, 256), 256, 0, R.st,
               (const CellT*)c->text, R.n, (const PosT*)ps_raw.p, j0, R.p, R.start_bits.p, R.end_bits, R.table.p, cap, R.slot_of_phrase.p, overflow);
}

template <class CellT>
void stage_dedup(Round& R) {
    grlgpu_ctx* c = R.c;
    const CellT* text = (const CellT*)c->text;
    // phrase numbering: per-tile popcounts of the start bitmap -> exclusive scan = index of a tile's first phrase
    constexpr int TW = fd_tile_words<CellT>();
    const u64 n_words = div_up(R.n, 32), n_tiles = div_up(n_words, TW);
    DevBuf<u32> tile_cnt(n_tiles, R.st);
    DevBuf<u64> tile_base(n_tiles, R.st), ptot(1, R.st);
    GRL_LAUNCH("tile_popc", R.n / 8, tile_popc_kernel, (unsigned)n_tiles, 256, 0, R.st, R.start_bits.p, n_words, TW, tile_cnt.p);
    exclusive_scan<u32, u64>(tile_cnt.p, tile_base.p, n_tiles, ptot.p, R.st);
    R.p = d2h_scalar(ptot.p, R.st);
    // function attributes are per device: set them for the current one on every call (a few microseconds), never cached process-wide
    GRL_CUDA(cudaFuncSetAttribute(dedup_cached_kernel<CellT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fd_smem_bytes<CellT>()));
    GRL_CUDA(cudaFuncSetAttribute(dedup_cached_kernel<CellT>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    const int n_sm = c->n_sm;
    const unsigned fd_grid = (unsigned)std::min<u64>(n_tiles, (u64)n_sm * FD_CTAS_PER_SM);  // persistent CTAs, tiles strided
    // the first tiles always run through the cached kernel and report how many phrases missed the caches;
    // the rest of the text takes the cached kernel (duplicate-heavy) or the thread-per-phrase kernel (unique-heavy)
    const bool force_uncached = (c->flags & GRLGPU_FLAG_FORCE_UNCACHED) != 0;
    const u64 t_pilot = force_uncached ? 0 : std::min<u64>(n_tiles, (c->flags & GRLGPU_FLAG_SMALL_PILOT) ? 1ull : 4ull * fd_grid);
    u64 j_pilot = R.p;
    if (t_pilot < n_tiles) j_pilot = t_pilot ? d2h_scalar(tile_base.p + t_pilot, R.st) : 0;
    BitmapCompactor bc;
    DevBuf<u8> ps_raw;
    bool counted = false;

    R.slot_of_phrase.alloc(R.p, R.st);
    DevBuf<u32> overflow(1, R.st);
    DevBuf<u64> stats(2, R.st);
    // capacity (any multiple of 256; slot = mulhi(hash, cap)). "full" = 1.6 p slots: load <= 0.625, the pass cannot
    // overflow (beyond 2^31 slots, i.e. p > 1.3e9: start at 2^28 and regrow on demand). A text long enough to have a
    // pilot starts SMALL instead (1.6 x the pilot's phrases): if the pilot says duplicate-heavy the dictionary is tiny
    // next to p and the small table is kept (no 30 GB init + occupancy scan for a 16 k-phrase dictionary); if it says
    // unique-heavy the pass restarts on the full table with the thread-per-phrase kernel.
    const u64 cap_max = (1ull << 31) - 256;
    const u64 want = std::max<u64>(1024, (R.p + R.p / 2 + R.p / 10 + 255) / 256 * 256);
    const u64 cap_full = want <= cap_max ? want : (1ull << 28);
    const bool has_rest = t_pilot < n_tiles;
    u64 cap = cap_full;
    if (t_pilot && has_rest) cap = std::min<u64>(cap_full, std::max<u64>(1ull << 20, (j_pilot + j_pilot / 2 + j_pilot / 10 + 255) / 256 * 256));
    if (c->flags & GRLGPU_FLAG_SMALL_TABLE) cap = 1024;
    int decided = has_rest ? (t_pilot ? -1 : 0) : 1;  // -1: ask the pilot, 1: cached kernel for the rest, 0: thread-per-phrase
    for (;;) {
        if (cap > cap_max) throw Error(GRLGPU_ERR_LIMIT, "phrase table would exceed 2^31 slots");
        R.table.alloc(cap, R.st);
        GRL_LAUNCH("table_init", cap * 16, table_init_kernel, grid_for(cap, 256), 256, 0, R.st, R.table.p, cap);
        overflow.zero();
        stats.zero();
        const bool run_pilot = t_pilot && decided != 0;
        if (run_pilot) {
            const u64 cells = std::min<u64>(R.n, t_pilot * TW * 32);
            GRL_LAUNCH("dedup_cached", cells * sizeof(CellT) + cells / 4 + j_pilot * 4, (dedup_cached_kernel<CellT>), fd_grid, FD_THREADS, fd_smem_bytes<CellT>(), R.st,
                       text, R.n, R.start_bits.p, R.end_bits, tile_base.p, (u64)0, t_pilot, R.table.p, cap, R.slot_of_phrase.p, overflow.p, stats.p);
        }
        if (has_rest) {
            if (decided == -1) {
                u64 hs[2];
                d2h_small(hs, stats.p, 16, R.st);
                GRL_CUDA(cudaStreamSynchronize(R.st));
                decided = hs[0] * 2 <= hs[1] ? 1 : 0;  // cached: at most half of the pilot's phrases had to go to the global table
                if (decided == 0 && cap < cap_full && !(c->flags & GRLGPU_FLAG_SMALL_TABLE)) { cap = cap_full; continue; }
            }
            if (decided == 1) {
                const u64 cells = R.n - t_pilot * TW * 32;
                GRL_LAUNCH("dedup_cached", cells * sizeof(CellT) + cells / 4 + (R.p - j_pilot) * 4, (dedup_cached_kernel<CellT>), fd_grid, FD_THREADS, fd_smem_bytes<CellT>(),
                           R.st, text, R.n, R.start_bits.p, R.end_bits, tile_base.p, t_pilot, n_tiles, R.table.p, cap, R.slot_of_phrase.p, overflow.p, (u64*)nullptr);
            } else {
                if (!counted) {
                    const u64 pc = bc.count(R.start_bits.p, R.n, R.st);
                    if (pc != R.p) throw Error(GRLGPU_ERR_STATE, "phrase count mismatch between tile counts and compaction");
                    counted = true;
                }
                const u64 j0 = run_pilot ? j_pilot : 0;
                if (R.n < (1ull << 31)) insert_uncached<CellT, u32>(R, bc, ps_raw, j0, cap, overflow.p);
                else insert_uncached<CellT, u64>(R, bc, ps_raw, j0, cap, overflow.p);
            }
        }
        bool ovf = d2h_scalar(overflow.p, R.st) != 0;
        u64 d = 0;
        if (!ovf) {
            DevBuf<u32> occ_bits(cap / 32, R.st);
            GRL_LAUNCH("table_occupancy", cap * 16, table_occupancy_kernel, (unsigned)(cap / 256), 256, 0, R.st, R.table.p, cap, occ_bits.p);
            BitmapCompactor oc;
            d = oc.count(occ_bits.p, cap, R.st);
            if (d * 10 <= cap * 7 || cap >= want) {  // load factor <= 0.7 (or the table can no longer be too small)
                R.occ_slots.alloc(d, R.st);
                oc.write<u32>(nullptr, R.occ_slots.p);
                R.d = d;
                R.cap = cap;
                break;
            }
        }
        if (cap >= cap_max) throw Error(GRLGPU_ERR_LIMIT, "phrase table would exceed 2^31 slots");
        const u64 grown = std::min<u64>(cap * 8, std::min<u64>(want, cap_max));  // too full: regrow and redo the pass
        cap = grown > cap ? grown : std::min<u64>(cap * 2, cap_max);              // (a probe-limit overflow at cap == want still has to grow)
    }
    ps_raw.release();
    R.ph_pos.alloc(R.d, R.st);
    R.ph_len.alloc(R.d, R.st);
    R.ph_freq.alloc(R.d, R.st);
    GRL_LAUNCH("dict_meta", 0, dict_meta_kernel, grid_for(R.d, 256), 256, 0, R.st, R.table.p, R.occ_slots.p, R.d, R.start_bits.p, R.end_bits, R.n, R.ph_pos.p, R.ph_len.p, R.ph_freq.p);
    dict_offsets(R);
    R.start_bits.release();
}

// phrase offsets inside the dictionary, number of entries, highest frequency, longest phrase
void dict_offsets(Round& R) {
    R.ph_off.alloc(R.d + 1, R.st);
    DevBuf<u64> tot64(1, R.st);
    {   // offsets as u64 first to detect overflow of the 32-bit entry index space
        DevBuf<u64> off64(R.d, R.st);
        exclusive_scan<u32, u64>(R.ph_len.p, off64.p, R.d, tot64.p, R.st);
        R.nE = d2h_scalar(tot64.p, R.st);
        if (R.nE >= 0xfffffff0ull) throw Error(GRLGPU_ERR_LIMIT, "dictionary of this round exceeds 2^32 symbols");
    }
    exclusive_scan<u32, u32>(R.ph_len.p, R.ph_off.p, R.d, R.ph_off.p + R.d, R.st);
    DevBuf<u64> mx(2, R.st);
    mx.zero();
    GRL_LAUNCH("reduce_max_u64", 0, reduce_max_u64_kernel, 296, 256, 0, R.st, R.ph_freq.p, R.d, mx.p);
    {
        DevBuf<u64> len64(R.d, R.st);
        GRL_LAUNCH("u32_to_u64", 0, u32_to_u64_kernel, grid_for(R.d, 256), 256, 0, R.st, R.ph_len.p, R.d, len64.p);
        GRL_LAUNCH("reduce_max_u64", 0, reduce_max_u64_kernel, 296, 256, 0, R.st, len64.p, R.d, mx.p + 1);
    }
    u64 hmx[2];
    d2h_small(hmx, mx.p, 16, R.st);
    R.max_freq = hmx[0];
    R.max_len = hmx[1];
}

template <class CellT, bool FIRST, class SymT>
void stage_gather(Round& R) {
    grlgpu_ctx* c = R.c;
    R.sym_bits = bit_width64(c->alphabet + 1);
    R.K = std::max(1, 64 / R.sym_bits);
    // refinement by key extension needs ceil((longest phrase + 1) / K) passes at most; beyond 64 passes (or when a test
    // forces it) the groups are refined by prefix doubling on position-based ranks instead
    R.ext_mode = !(c->flags & GRLGPU_FLAG_FORCE_DOUBLING) && (R.max_len + 1 + (u64)R.K - 1) / (u64)R.K <= 64;
    R.spare = (R.ext_mode && R.sym_bits * R.K < 64) ? 64 - R.sym_bits * R.K : 0;
    const CellT* text = (const CellT*)c->text;
    DevBuf<u32> voff;
    R.nS = R.nE;
    if (R.ext_mode) {
        voff.alloc(R.d + 1, R.st);
        DevBuf<u32> tot(1, R.st);
        IsSuffix isuf0{c->is_suffix.p, c->sep, c->first};
        GRL_LAUNCH("phrase_vlen", R.d * 48, (phrase_vlen_kernel<CellT, FIRST>), grid_for(R.d, 256), 256, 0, R.st, text, R.ph_pos.p, R.ph_len.p, R.d, isuf0, voff.p);
        exclusive_scan<u32, u32>(voff.p, voff.p, R.d, voff.p + R.d, R.st);
        R.nS = d2h_scalar(voff.p + R.d, R.st);
        R.keys.alloc(R.nS, R.st);
        R.vals.alloc(R.nS, R.st);
    }
    R.D_raw.alloc((R.nE + 1) * sizeof(SymT), R.st);
    if (R.c->flags & GRLGPU_FLAG_KEEP_DICT) R.phr_of.alloc(R.nE, R.st);  // only the test hooks read it
    R.rem.alloc(R.nE, R.st);
    R.einfo.alloc(R.nE, R.st);
    IsSuffix isuf{R.c->is_suffix.p, R.c->sep, R.c->first};
    // metasymbols go to the phrase's table slot
    GRL_LAUNCH("dict_gather", R.nE * (sizeof(CellT) + sizeof(SymT) + 20) + R.nS * 12 + R.d * 32, (dict_gather_kernel<CellT, FIRST, SymT>), grid_for(R.d, 256), 256, 0, R.st, text,
               R.ph_pos.p, R.ph_len.p, R.ph_off.p, R.ph_freq.p, R.occ_slots.p, R.d, isuf, (SymT*)R.D_raw.p, R.phr_of.p, R.rem.p,
               R.einfo.p, (const u32*)voff.p, c->alphabet + 1, R.sym_bits, R.K, R.spare, R.keys.p, R.vals.p);
}

// One refinement depth of the suffix order: the active elements (slot j: extension key nk[j], gflag[j] = first of its group)
// are sorted by key inside their groups. -> perm[q] = active index of the element that belongs at slot q, flags[q] = 1 where
// a new (sub)group starts. Tile-local segmented sort for the groups that fit a window; the flagged rest goes through two
// device-wide radix sorts (by key, then stably by group).
void refine_sort_groups(cudaStream_t st, const u64* nk, const u32* gflag, u64 nA, int key_bits, DevBuf<u32>& perm, DevBuf<u32>& flags) {
    perm.alloc(nA, st);
    flags.alloc(nA, st);
    if (nA == 0) return;
    DevBuf<u32> lflag(nA, st), lexcl(nA, st), cnt(1, st);
    GRL_LAUNCH("ext_local_sort", nA * 24, ext_local_sort_kernel, (unsigned)div_up(nA, LS_WIN), LS_THREADS, 0, st, nk, gflag, nA, perm.p, flags.p, lflag.p);
    exclusive_scan<u32, u32>(lflag.p, lexcl.p, nA, cnt.p, st);
    const u64 nLft = d2h_scalar(cnt.p, st);
    if (getenv("GRLGPU_TRACE")) fprintf(stderr, "[grlgpu]   refine sort: %llu active, %llu through the device-wide path\n", nA, nLft);
    if (nLft == 0) return;
    DevBuf<u32> lpos(nLft, st), lv(nLft, st), lv_alt(nLft, st), lg(nLft, st), gexcl(nLft, st), lf(nLft, st);
    DevBuf<u64> lk(nLft, st), lk_alt(nLft, st), lnk(nLft, st);
    GRL_LAUNCH("ext_left_gather", nA * 8 + nLft * 32, ext_left_gather_kernel, grid_for(nA, 256), 256, 0, st, lflag.p, lexcl.p, nk, gflag, nA, lpos.p, lk.p, lnk.p, lv.p, lg.p);
    exclusive_scan<u32, u32>(lg.p, gexcl.p, nLft, cnt.p, st);
    const u64 n_groups = d2h_scalar(cnt.p, st);
    u64 *kp = lk.p, *ka = lk_alt.p;
    u32 *vp = lv.p, *va = lv_alt.p;
    radix_sort_pairs(&kp, &vp, &ka, &va, nLft, key_bits, st);  // by the extension key ...
    GRL_LAUNCH("ext_gid", nLft * 12, ext_gid_kernel, grid_for(nLft, 256), 256, 0, st, lg.p, gexcl.p, nLft);
    GRL_LAUNCH("ext_group_keys", nLft * 16, ext_group_keys_kernel, grid_for(nLft, 256), 256, 0, st, vp, gexcl.p, nLft, kp);
    radix_sort_pairs(&kp, &vp, &ka, &va, nLft, std::max(1, bit_width64(n_groups)), st);  // ... then, stably, by group
    GRL_LAUNCH("ext_heads", nLft * 24, ext_heads_kernel, grid_for(nLft, 256), 256, 0, st, vp, kp, lnk.p, nLft, lf.p);
    GRL_LAUNCH("ext_left_scatter", nLft * 20, ext_left_scatter_kernel, grid_for(nLft, 256), 256, 0, st, lpos.p, vp, lf.p, nLft, perm.p, flags.p);
    GRL_CUDA(cudaStreamSynchronize(st));  // the temporaries above go back to the pool
}

// ---------------- dictionary stage: suffix order, groups, ranks, pre-BWT, rules, metasymbols ----------------
template <class SymT>
void stage_dict(Round& R) {
    grlgpu_ctx* c = R.c;
    cudaStream_t st = R.st;
    const u64 nE = R.nE, A = c->alphabet;
    const SymT* D = (const SymT*)R.D_raw.p;
    IsSuffix isuf{c->is_suffix.p, c->sep, c->first};

    // -- suffix order: one full sort on the packed first key, then refinement of the unresolved groups only --
    const bool ext_mode = R.ext_mode;
    const u64 nS = R.nS;  // sorted items: the valid entries (key extension) or every entry (prefix doubling)
    const u64 n_words = div_up(nS, 32);
    DevBuf<u32> order_buf, head_bits(n_words, st);
    u64 G = 0;
    {
        DevBuf<u64> keys = std::move(R.keys), keys_alt(nS, st);
        DevBuf<u32> vals = std::move(R.vals), vals_alt(nS, st);
        const int sym_bits = R.sym_bits, K = R.K;
        if (!ext_mode) {
            keys.alloc(nS, st);
            vals.alloc(nS, st);
            GRL_LAUNCH("sfx_first_key", nE * (sizeof(SymT) + 4 + 12), (sfx_first_key_kernel<SymT>), grid_for(nE, 256), 256, 0, st, D, R.rem.p, nE, A + 1, sym_bits, K, keys.p, vals.p);
        }
        u64 *kp = keys.p, *ka = keys_alt.p;
        u32 *vp = vals.p, *va = vals_alt.p;
        radix_sort_pairs(&kp, &vp, &ka, &va, nS, std::min(64, sym_bits * K + R.spare), st);
        if (vp != vals.p) std::swap(vals, vals_alt);
        order_buf = std::move(vals);
        vals_alt.release();
        u32* order_w = order_buf.p;
        u64 nA = 0;
        DevBuf<u32> apos;
        if (ext_mode) {
            {
                DevBuf<u32> flags(nS, st), active_bits(n_words, st);
                GRL_LAUNCH("first_heads", nS * 12, first_heads_kernel, grid_for(nS, 256), 256, 0, st, kp, nS, sym_bits, R.spare, A + 1, flags.p, head_bits.p, active_bits.p);
                keys.release(); keys_alt.release();
                BitmapCompactor ac;
                nA = ac.count(active_bits.p, nS, st);
                apos.alloc(nA, st);
                if (nA) ac.write<u32>(nullptr, apos.p);
            }
            u64 dpt = (u64)K;  // codes already compared
            while (nA > 0) {
                if (dpt > R.max_len + 1) throw Error(GRLGPU_ERR_STATE, "suffix refinement did not converge");
                DevBuf<u64> nk(nA, st);
                DevBuf<u32> ev(nA, st), gflag(nA, st), excl(nA, st), cnt(1, st), perm, flags;
                GRL_LAUNCH("ext_keys", nA * 32, (ext_keys_kernel<SymT>), grid_for(nA, 256), 256, 0, st, apos.p, order_w, D, R.rem.p, head_bits.p, nA, dpt, A + 1, sym_bits, K,
                           (u64*)nullptr, (u32*)nullptr, nk.p, ev.p, gflag.p);
                if (getenv("GRLGPU_TRACE")) fprintf(stderr, "[grlgpu] round %d refine: depth %llu, active %llu (of %llu sorted)\n", c->round + 1, dpt, nA, nS);
                refine_sort_groups(st, nk.p, gflag.p, nA, std::min(64, sym_bits * K), perm, flags);
                const u32* avp = perm.p;
                GRL_LAUNCH("ext_writeback", nA * 16, ext_writeback_kernel, grid_for(nA, 256), 256, 0, st, apos.p, avp, ev.p, flags.p, nA, order_w, head_bits.p);
                dpt += (u64)K;
                GRL_LAUNCH("ext_next", nA * 16, ext_next_kernel, grid_for(nA, 256), 256, 0, st, apos.p, avp, ev.p, head_bits.p, R.rem.p, nA, nS, dpt, flags.p);
                exclusive_scan<u32, u32>(flags.p, excl.p, nA, cnt.p, st);
                const u64 nA2 = d2h_scalar(cnt.p, st);
                DevBuf<u32> apos2(nA2, st);
                if (nA2) GRL_LAUNCH("compact_apos", nA * 12, compact_apos_kernel, grid_for(nA, 256), 256, 0, st, flags.p, excl.p, apos.p, nA, apos2.p);
                apos = std::move(apos2);
                nA = nA2;
            }
        } else {
        R.rank.alloc(nE, st);
        {   // heads, position-based ranks and the first active set
            DevBuf<u32> flags(nE, st), excl(nE, st), active_bits(n_words, st), gcount(1, st);
            GRL_LAUNCH("first_heads", nE * 12, first_heads_kernel, grid_for(nE, 256), 256, 0, st, kp, nE, sym_bits, 0, A + 1, flags.p, head_bits.p, active_bits.p);
            keys.release(); keys_alt.release();
            exclusive_scan<u32, u32>(flags.p, excl.p, nE, gcount.p, st);
            const u64 G0 = d2h_scalar(gcount.p, st);
            DevBuf<u32> head_pos(G0, st);
            GRL_LAUNCH("head_pos", nE * 8, head_pos_kernel, grid_for(nE, 256), 256, 0, st, flags.p, excl.p, (const u32*)nullptr, nE, head_pos.p);
            if (nE <= (1ull << 24)) {  // the whole rank array fits the L2: scatter directly
                GRL_LAUNCH("assign_hrank", nE * 20, assign_hrank_kernel, grid_for(nE, 256), 256, 0, st, flags.p, excl.p, head_pos.p, order_w, nE, R.rank.p);
            } else {
                // a random 4-byte scatter over GBs costs ~78 B of DRAM traffic per entry (sector read-modify-write); partition the
                // (entry, rank) pairs by the entry's top byte first, so that every stretch of pairs lands in one 64 MB window
                DevBuf<u32> pk(nE, st), pv(nE, st), pk2(nE, st), pv2(nE, st);
                GRL_LAUNCH("hrank_pairs", nE * 20, hrank_pairs_kernel, grid_for(nE, 256), 256, 0, st, flags.p, excl.p, head_pos.p, order_w, nE, pk.p, pv.p);
                u32 *k1 = pk.p, *v1 = pv.p, *k2 = pk2.p, *v2 = pv2.p;
                radix_partition_u32(&k1, &v1, &k2, &v2, nE, 24, st);
                GRL_LAUNCH("scatter_pairs", nE * 12, scatter_pairs_kernel, grid_for(nE, 256), 256, 0, st, k1, v1, nE, R.rank.p);
            }
            BitmapCompactor ac;
            nA = ac.count(active_bits.p, nE, st);
            apos.alloc(nA, st);
            if (nA) ac.write<u32>(nullptr, apos.p);
        }
        const int rb = bit_width64(nE + 1);
        u64 h = (u64)K;
        while (nA > 0) {  // a key of h codes covers any suffix (<= max_len symbols + terminator) once h > max_len
            if (h > R.max_len + 1) throw Error(GRLGPU_ERR_STATE, "suffix refinement did not converge");
            DevBuf<u64> ak(nA, st), ak_alt(nA, st);
            DevBuf<u32> av(nA, st), av_alt(nA, st), flags(nA, st), excl(nA, st), cnt(1, st);
            u64 *akp = ak.p, *aka = ak_alt.p;
            u32 *avp = av.p, *ava = av_alt.p;
            GRL_LAUNCH("active_keys", nA * 36, active_keys_kernel, grid_for(nA, 256), 256, 0, st, apos.p, order_w, R.rank.p, R.rem.p, nA, h, (u32)(nE + 1), rb, akp, avp);
            radix_sort_pairs(&akp, &avp, &aka, &ava, nA, 2 * rb, st);
            GRL_LAUNCH("key_head_flags", nA * 12, key_head_flags_kernel, grid_for(nA, 256), 256, 0, st, akp, nA, flags.p);
            exclusive_scan<u32, u32>(flags.p, excl.p, nA, cnt.p, st);
            const u64 nH = d2h_scalar(cnt.p, st);
            DevBuf<u32> head_pos(nH, st);
            GRL_LAUNCH("head_pos", nA * 12, head_pos_kernel, grid_for(nA, 256), 256, 0, st, flags.p, excl.p, apos.p, nA, head_pos.p);
            GRL_LAUNCH("assign_hrank", nA * 20, assign_hrank_kernel, grid_for(nA, 256), 256, 0, st, flags.p, excl.p, head_pos.p, avp, nA, R.rank.p);
            GRL_LAUNCH("refine_writeback", nA * 16, refine_writeback_kernel, grid_for(nA, 256), 256, 0, st, apos.p, avp, flags.p, nA, order_w, head_bits.p);
            h *= 2;
            GRL_LAUNCH("active_next", nA * 16, active_next_kernel, grid_for(nA, 256), 256, 0, st, apos.p, avp, head_bits.p, R.rem.p, nA, nE, h, flags.p);
            exclusive_scan<u32, u32>(flags.p, excl.p, nA, cnt.p, st);
            const u64 nA2 = d2h_scalar(cnt.p, st);
            DevBuf<u32> apos2(nA2, st);
            if (nA2) GRL_LAUNCH("compact_apos", nA * 12, compact_apos_kernel, grid_for(nA, 256), 256, 0, st, flags.p, excl.p, apos.p, nA, apos2.p);
            apos = std::move(apos2);
            nA = nA2;
        }
            }  // doubling
    }
    const u32* order = order_buf.p;
    // dense group ids from the head bitmap: per-word prefix counts
    DevBuf<u32> head_pref(n_words, st);
    {
        DevBuf<u32> wc(n_words, st), gtot(1, st);
        GRL_LAUNCH("popc_words", n_words * 8, popc_words_kernel, grid_for(n_words, 256), 256, 0, st, head_bits.p, n_words, wc.p);
        exclusive_scan<u32, u32>(wc.p, head_pref.p, n_words, gtot.p, st);
        G = d2h_scalar(gtot.p, st);
    }
    R.G = G;

    // -- group aggregates --
    DevBuf<u32> gcnt(G, st), grep(G, st), ghead(G, st), rflag(G, st), vflag(G, st), rrank(G, st), vidx(G, st);
    DevBuf<u64> gacc(G, st), gmin(G, st), gmax(G, st), psym(G, st), gfull(G, st);
    gcnt.zero(); gacc.zero(); gmax.zero(); gmin.fill_ff();
    GRL_LAUNCH("group_reduce", nS * 24 + G * 32, group_reduce_kernel, grid_for(nS, 256), 256, 0, st, order, head_bits.p, head_pref.p, R.einfo.p, nS, gcnt.p, gacc.p, gmin.p, gmax.p, grep.p, ghead.p, gfull.p);
    R.einfo.release();
    const u64 bwt_dummy = A + 1, hocc_dummy = A + 2;  // exact_par_phase.hpp:113-115
    GRL_LAUNCH("group_finalize", 0, group_finalize_kernel, grid_for(G, 256), 256, 0, st, gcnt.p, gmin.p, gmax.p, G, bwt_dummy, hocc_dummy, rflag.p, vflag.p, psym.p);
    DevBuf<u32> cnt2(2, st);
    exclusive_scan<u32, u32>(rflag.p, rrank.p, G, cnt2.p, st);
    exclusive_scan<u32, u32>(vflag.p, vidx.p, G, cnt2.p + 1, st);
    u32 hc[2];
    d2h_small(hc, cnt2.p, 8, st);
    const u64 tot = hc[0], nV = hc[1];
    if (tot >= (1ull << 30)) throw Error(GRLGPU_ERR_LIMIT, "more than 2^30 ranks in one round");
    R.tot = tot;

    // -- preliminary BWT: maximal runs over the valid groups --
    DevLevel& L = c->lvl;
    L.sym_bytes = sizeof(SymT);
    {
        DevBuf<u64> csym(nV, st), clen(nV, st);
        GRL_LAUNCH("prebwt_compact", 0, prebwt_compact_kernel, grid_for(G, 256), 256, 0, st, vflag.p, vidx.p, psym.p, gacc.p, G, csym.p, clen.p);
        DevBuf<u32> hflag(nV, st), hexcl(nV, st), nrun(1, st);
        GRL_LAUNCH("key_head_flags", 0, key_head_flags_kernel, grid_for(nV, 256), 256, 0, st, csym.p, nV, hflag.p);
        exclusive_scan<u32, u32>(hflag.p, hexcl.p, nV, nrun.p, st);
        R.n_pre = d2h_scalar(nrun.p, st);
        L.pre_sym.alloc(R.n_pre * sizeof(SymT), st);
        L.pre_len.alloc(R.n_pre, st);
        L.pre_len.zero();
        GRL_LAUNCH("prebwt_runs", 0, (prebwt_runs_kernel<SymT>), grid_for(nV, 256), 256, 0, st, csym.p, clen.p, hflag.p, hexcl.p, nV, (SymT*)L.pre_sym.p, L.pre_len.p);
    }

    // -- metasymbols, next is_suffix, hocc marks, rules --
    DevBuf<u8> is_suffix_next(tot, st);
    is_suffix_next.zero();
    DevBuf<u32> erank(nE, st);
    erank.fill_ff();
    GRL_LAUNCH("full_apply", G * 20 + R.d * 40, full_apply_kernel, grid_for(G, 256), 256, 0, st, gcnt.p, rflag.p, rrank.p, gfull.p, G, R.table.p, is_suffix_next.p);
    gfull.release();
    if (ext_mode) {  // hocc marks in sorted order: group info is read sequentially, entries need no rank of their own
        DevBuf<u32> ginfo(G, st);
        GRL_LAUNCH("pack_ginfo_dense", G * 16, pack_ginfo_dense_kernel, grid_for(G, 256), 256, 0, st, gcnt.p, rflag.p, rrank.p, G, ginfo.p);
        GRL_LAUNCH("group_apply", nS * 12, group_apply_kernel, grid_for(nS, 256), 256, 0, st, order, head_bits.p, head_pref.p, ginfo.p, nS, erank.p);
    } else {
        DevBuf<u32> ginfo(nE, st);  // indexed by head position
        GRL_LAUNCH("pack_ginfo", G * 20, pack_ginfo_kernel, grid_for(G, 256), 256, 0, st, gcnt.p, rflag.p, rrank.p, ghead.p, G, ginfo.p);
        GRL_LAUNCH("entry_finalize", nE * 12, entry_finalize_kernel, grid_for(nE, 256), 256, 0, st, R.rank.p, nE, ginfo.p, erank.p);
    }
    L.rule_l.alloc(tot * sizeof(SymT), st);
    L.rule_r.alloc(tot * sizeof(SymT), st);
    L.has_hocc.alloc(tot, st);
    const u64 alph3 = A + 3, metasym_dummy = alph3 + tot + 1;  // exact_par_phase.cpp:19-20
    // model: 16 B of sequential group records + three random 32-byte sectors per ranked group (rem, hocc mark, symbols of the representative)
    // + the rule written (2 symbols + 1 byte)
    GRL_LAUNCH("rules", G * 16 + tot * (96 + 2 * sizeof(SymT) + 1), (rules_kernel<SymT>), grid_for(G, 256), 256, 0, st, gcnt.p, rflag.p, rrank.p, grep.p, G, D, R.rem.p, erank.p, isuf, alph3, metasym_dummy, (SymT*)L.rule_l.p, (SymT*)L.rule_r.p, L.has_hocc.p);
    L.tot = tot;
    L.n_pre = R.n_pre;
    // every valid dictionary entry contributes its phrase's frequency to exactly one run: the lengths of a level sum to at most
    // n + p (phrases overlap by one cell)
    c->lvl_n_in = R.n + R.p;

    if (c->flags & GRLGPU_FLAG_KEEP_DICT) {
        c->kd_d = R.d; c->kd_nE = nE; c->kd_nS = nS;
        c->kd_order.alloc(nS, st);
        GRL_CUDA(cudaMemcpyAsync(c->kd_order.p, order, nS * 4, cudaMemcpyDeviceToDevice, st));
    }
    GRL_CUDA(cudaStreamSynchronize(st));  // temporaries above are released in stream order
    c->is_suffix = std::move(is_suffix_next);
}

template <class OutT>
void stage_rewrite(Round& R, DevBuf<u8>& new_text, DevBuf<u32>& new_end_bits) {
    new_text.alloc(std::max<u64>(R.p * sizeof(OutT), 16), R.st);
    new_end_bits.alloc(div_up(R.p, 32), R.st);
    GRL_LAUNCH("rewrite", R.p * (4 + 16 + sizeof(OutT)), (rewrite_kernel<OutT>), grid_for(R.p, 256), 256, 0, R.st, R.slot_of_phrase.p, R.p, R.table.p, (OutT*)new_text.p, new_end_bits.p);
}

// rewrite the local text with the metasymbols now stored in the local table, report, and make the parse
// the text of the next round. `tot` / `n_pre` / dictionary sizes describe the round's (global) dictionary.
struct RoundTimes { float all = 0, text = 0, dict = 0; };
void finish_round(grlgpu_ctx* c, Round& R, u64 tot, u64 n_pre, u64 dict_d, u64 dict_nE, u64 max_freq, const RoundTimes& tm, Timer* t_all, grlgpu_round_t* out) {
    Timer t_rw(c->st);
    t_rw.start();
    const int bps = bit_width64(tot) + 1;  // exact_par_phase.cpp:456-465
    const int w_out = bps <= 8 ? 1 : bps <= 16 ? 2 : bps <= 32 ? 4 : 8;
    DevBuf<u8> new_text;
    DevBuf<u32> new_end;
    if (w_out == 1) stage_rewrite<u8>(R, new_text, new_end);
    else if (w_out == 2) stage_rewrite<u16>(R, new_text, new_end);
    else if (w_out == 4) stage_rewrite<u32>(R, new_text, new_end);
    else stage_rewrite<u64>(R, new_text, new_end);
    t_rw.stop();
    if (t_all) t_all->stop();

    memset(out, 0, sizeof(*out));
    out->round = (u64)c->round + 1;
    out->n_in = R.n;
    out->n_strings = c->n_strings;
    out->parse_len = R.p;
    out->n_phrases = dict_d;
    out->dict_syms = dict_nE;
    out->max_freq = max_freq;
    out->alphabet = c->alphabet;
    out->tot_phrases = tot;
    out->n_pre_runs = n_pre;
    out->cell_bytes_in = (u32)c->w;
    out->cell_bytes_out = (u32)w_out;
    out->sym_bytes = (u32)c->lvl.sym_bytes;
    out->done = R.p == c->n_strings;
    out->algorithmic_bytes = R.n * (u64)c->w + R.p * (u64)w_out + dict_nE * (u64)c->w + 8 * dict_d;
    out->device_ms = t_all ? t_all->ms() : tm.all;
    out->text_pass_ms = tm.text;
    out->dict_ms = tm.dict;
    out->rewrite_ms = t_rw.ms();

    if ((c->flags & GRLGPU_FLAG_KEEP_DICT) && c->kd_meta.p) {  // metasymbol per distinct phrase, for tests
        std::vector<u32> slots(R.d);
        GRL_CUDA(cudaMemcpy(slots.data(), R.occ_slots.p, R.d * 4, cudaMemcpyDeviceToHost));
        std::vector<ulonglong2> tab(R.cap);
        GRL_CUDA(cudaMemcpy(tab.data(), R.table.p, R.cap * sizeof(ulonglong2), cudaMemcpyDeviceToHost));
        std::vector<u64> metas(R.d);
        for (u64 i = 0; i < R.d; i++) metas[i] = tab[slots[i]].y;
        GRL_CUDA(cudaMemcpy(c->kd_meta.p, metas.data(), R.d * 8, cudaMemcpyHostToDevice));
    }

    // the parse becomes the text of the next round
    GRL_CUDA(cudaStreamSynchronize(c->st));
    c->prof.resolve();
    c->text_own = std::move(new_text);
    c->text = c->text_own.p;
    c->end_bits = std::move(new_end);
    c->n = R.p;
    c->w = w_out;
    c->first = false;
    c->lvl_alphabet = c->alphabet;  // A of the round that produced the level (the induction needs it: dummies A+1 / A+2, rules from A+3)
    c->alphabet = tot;
    c->round++;
    c->done = out->done != 0;
}

template <class CellT, bool FIRST>
void run_round_t(grlgpu_ctx* c, grlgpu_round_t* out) {
    Round R(c);
    Timer t_all(c->st), t_text(c->st), t_dict(c->st);
    t_all.start();
    t_text.start();
    stage_flags<CellT, FIRST>(R);
    stage_dedup<CellT>(R);
    t_text.stop();
    t_dict.start();
    const u64 A = c->alphabet;
    // rule values go up to A + 3 + tot + 1 with tot <= nE
    const bool wide = (A + R.nE + 8) >= (1ull << 32);
    if (wide) { stage_gather<CellT, FIRST, u64>(R); stage_dict<u64>(R); }
    else { stage_gather<CellT, FIRST, u32>(R); stage_dict<u32>(R); }
    t_dict.stop();
    if (c->flags & GRLGPU_FLAG_KEEP_DICT) {
        c->kd_D = std::move(R.D_raw);
        c->kd_off = std::move(R.ph_off);
        c->kd_len = std::move(R.ph_len);
        c->kd_freq = std::move(R.ph_freq);
        c->kd_phr_of = std::move(R.phr_of);
        c->kd_meta.alloc(R.d, c->st);
    }
    RoundTimes tm;
    tm.text = t_text.ms();
    tm.dict = t_dict.ms();
    finish_round(c, R, R.tot, R.n_pre, R.d, R.nE, R.max_freq, tm, &t_all, out);
}

#include "mg2.cuh"
#include "induce.cuh"
#include "invert.cuh"
#include "fm.cuh"

void run_round(grlgpu_ctx* c, grlgpu_round_t* out) {
    if (c->first) {
        switch (c->w) {
            case 1: run_round_t<u8, true>(c, out); break;
            case 2: run_round_t<u16, true>(c, out); break;
            case 4: run_round_t<u32, true>(c, out); break;
            default: run_round_t<u64, true>(c, out); break;
        }
    } else {
        switch (c->w) {
            case 1: run_round_t<u8, false>(c, out); break;
            case 2: run_round_t<u16, false>(c, out); break;
            case 4: run_round_t<u32, false>(c, out); break;
            default: run_round_t<u64, false>(c, out); break;
        }
    }
}

template <class CellT>
void compute_stats(grlgpu_ctx* c) {
    const CellT* text = (const CellT*)c->text;
    CellT sep_c;
    GRL_CUDA(cudaMemcpyAsync(&sep_c, text + (c->n - 1), sizeof(CellT), cudaMemcpyDeviceToHost, c->st));
    GRL_CUDA(cudaStreamSynchronize(c->st));
    DevBuf<StatsAcc> acc(1, c->st);
    StatsAcc h;
    memset(&h, 0, sizeof(h));
    h.min_sym = ~0ULL;
    GRL_CUDA(cudaMemcpyAsync(acc.p, &h, sizeof(h), cudaMemcpyHostToDevice, c->st));
    GRL_LAUNCH("stats", 0, (stats_kernel<CellT>), 148 * 8, 256, 0, c->st, text, c->n, sep_c, acc.p);
    GRL_CUDA(cudaMemcpyAsync(&h, acc.p, sizeof(h), cudaMemcpyDeviceToHost, c->st));
    GRL_CUDA(cudaStreamSynchronize(c->st));
    grlgpu_stats_t& s = c->stats;
    s.n_syms = c->n;
    s.sep_sym = (u64)sep_c;
    s.n_strings = h.n_sep;
    s.max_sym_freq = c->n;  // utils.cpp:117
    if (sizeof(CellT) == 1) {  // utils.cpp:161-175
        memcpy(c->hist, h.hist, sizeof(c->hist));
        int lo = 0, hi = 255;
        while (h.hist[lo] == 0) lo++;
        while (h.hist[hi] == 0) hi--;
        s.min_sym = lo; s.max_sym = hi;
        u64 m = 0;
        for (int i = 0; i < 256; i++) m = std::max<u64>(m, h.hist[i]);
        s.max_sym_freq = m;
    } else { s.min_sym = h.min_sym; s.max_sym = h.max_sym; }
    if (s.sep_sym != s.min_sym) throw Error(GRLGPU_ERR_ILL_FORMED, "the collection is ill formed: the last symbol is not the smallest symbol");
    // longest string: positions of the separators -> adjacent differences
    {
        const u64 n_words = div_up(c->n, 32);
        DevBuf<u32> eb(n_words, c->st), sb(n_words, c->st);
        GRL_LAUNCH("first_round_end_bits", c->n * sizeof(CellT), (first_round_end_bits_kernel<CellT>), grid_for(n_words, 256), 256, 0, c->st, text, c->n, sep_c, eb.p);
        GRL_LAUNCH("next_start_bits", 0, next_start_bits_kernel, grid_for(n_words, 256), 256, 0, c->st, eb.p, c->n, sb.p);
        BitmapCompactor bc;
        const u64 ns = bc.count(sb.p, c->n, c->st);
        DevBuf<u64> ptrs(ns + 1, c->st), mx(1, c->st);
        bc.write<u64>(nullptr, ptrs.p);
        GRL_CUDA(cudaMemcpyAsync(ptrs.p + ns, &c->n, 8, cudaMemcpyHostToDevice, c->st));
        mx.zero();
        GRL_LAUNCH("adjacent_max_diff", 0, adjacent_max_diff_kernel, 296, 256, 0, c->st, ptrs.p, ns, mx.p);
        s.longest_string = d2h_scalar(mx.p, c->st);
    }
    c->sep = s.sep_sym;
    c->n_strings = s.n_strings;
    c->alphabet = s.max_sym + 1;  // exact_par_phase.cpp:316
    c->have_stats = true;
}

// order-insensitive digests of a level's artefacts: sums mod 2^64 that add up across per-rank slices of the same level
// (rules weighted by their GLOBAL rank, preliminary-BWT runs by symbol so that a run split at a slice seam counts the same)
template <class SymT>
static __global__ void __launch_bounds__(256) level_checksum_kernel(const SymT* __restrict__ rule_l, const SymT* __restrict__ rule_r, const u8* __restrict__ has_hocc, u64 tot,
                                                                    u64 rank_base, const SymT* __restrict__ pre_sym, const u64* __restrict__ pre_len, u64 n_pre, u64* acc) {
    u64 a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (u64)gridDim.x * blockDim.x) {
        const u64 u = rank_base + i + 1;
        a0 += u * (((u64)rule_l[i] * 0x9E3779B97F4A7C15ULL) ^ ((u64)rule_r[i] * 0xC2B2AE3D27D4EB4FULL));
        a1 += u * (u64)has_hocc[i];
    }
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_pre; i += (u64)gridDim.x * blockDim.x) {
        a2 += pre_len[i];
        a3 += ((u64)pre_sym[i] * 0x9E3779B97F4A7C15ULL + 1) * pre_len[i];
    }
    a0 = warp_sum(a0); a1 = warp_sum(a1); a2 = warp_sum(a2); a3 = warp_sum(a3);
    if (lane_id() == 0) { atomicAdd(&acc[0], a0); atomicAdd(&acc[1], a1); atomicAdd(&acc[2], a2); atomicAdd(&acc[3], a3); }
}
inline void level_checksum(cudaStream_t st, const LevelView& v, u64* host_out4) {
    DevBuf<u64> acc(4, st);
    acc.zero();
    if (v.sym_bytes == 8)
        GRL_LAUNCH("level_checksum", 0, (level_checksum_kernel<u64>), 296, 256, 0, st, (const u64*)v.rule_l, (const u64*)v.rule_r, v.has_hocc, v.tot, v.rank_base, (const u64*)v.pre_sym,
                   v.pre_len, v.n_pre, acc.p);
    else
        GRL_LAUNCH("level_checksum", 0, (level_checksum_kernel<u32>), 296, 256, 0, st, (const u32*)v.rule_l, (const u32*)v.rule_r, v.has_hocc, v.tot, v.rank_base, (const u32*)v.pre_sym,
                   v.pre_len, v.n_pre, acc.p);
    d2h_small(host_out4, acc.p, 32, st);
}

inline void ensure_stats(grlgpu_ctx* ctx) {
    if (ctx->have_stats) return;
    switch (ctx->w) {
        case 1: compute_stats<u8>(ctx); break;
        case 2: compute_stats<u16>(ctx); break;
        case 4: compute_stats<u32>(ctx); break;
        default: compute_stats<u64>(ctx); break;
    }
}

thread_local std::string t_last_error;  // errors of calls that have no context (communicator creation): grlgpu_last_error(NULL)
template <class F>
int guarded(grlgpu_ctx* c, F&& f) {
    struct CtxGuard {  // per-call binding of the context's launch accounting and memory pool
        // GRLGPU_NO_POOL=1 (compute-sanitizer runs): every buffer is its own cudaMalloc, so memcheck sees the true bounds
        explicit CtxGuard(grlgpu_ctx* x) { g_prof = x ? &x->prof : nullptr; g_pool = (x && !no_pool()) ? &x->pool : nullptr; }
        static bool no_pool() { static const bool v = getenv("GRLGPU_NO_POOL") != nullptr; return v; }
        ~CtxGuard() { g_prof = nullptr; g_pool = nullptr; }
    } cg(c);
    try {
        if (c) GRL_CUDA(cudaSetDevice(c->device));
        f();
        return GRLGPU_OK;
    } catch (const Error& e) {
        if (c) c->last_error = e.what(); else t_last_error = e.what();
        cudaGetLastError();
        if (e.code == GRLGPU_ERR_CUDA && std::string(e.what()).find("out of memory") != std::string::npos) return GRLGPU_ERR_NOMEM;
        return e.code;
    } catch (const std::exception& e) {
        if (c) c->last_error = e.what(); else t_last_error = e.what();
        return GRLGPU_ERR_CUDA;
    }
}

}  // namespace

struct grlgpu_comm { std::unique_ptr<grl::Comm> c; };
struct grlgpu_local_group {
    grl::LocalGroup g;
    explicit grlgpu_local_group(int w) : g(w) {}
};

extern "C" {

int grlgpu_create_on_stream(grlgpu_ctx** ctx, int device, uint64_t flags, void* cuda_stream);
int grlgpu_create(grlgpu_ctx** ctx, int device, uint64_t flags) { return grlgpu_create_on_stream(ctx, device, flags, nullptr); }

int grlgpu_create_on_stream(grlgpu_ctx** ctx, int device, uint64_t flags, void* cuda_stream) {
    if (!ctx) return GRLGPU_ERR_ARG;
    *ctx = nullptr;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0 || device < 0 || device >= n_dev) return GRLGPU_ERR_CUDA;
    std::unique_ptr<grlgpu_ctx> c(new grlgpu_ctx());
    c->device = device;
    c->flags = flags;
    int rc = guarded(c.get(), [&] {
        c->pool.init(device);
        GRL_CUDA(cudaDeviceGetAttribute(&c->n_sm, cudaDevAttrMultiProcessorCount, device));
        if (cuda_stream) { c->st = (cudaStream_t)cuda_stream; c->own_stream = false; }
        else GRL_CUDA(cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking));
    });
    if (rc != GRLGPU_OK) return rc;
    *ctx = c.release();
    return GRLGPU_OK;
}

uint64_t grlgpu_trim(void) {
    DevicePool tmp;
    try {
        DevicePool::resolve("cuMemUnmap", tmp.p_unmap); DevicePool::resolve("cuMemRelease", tmp.p_release); DevicePool::resolve("cuMemAddressFree", tmp.p_addrfree);
    } catch (const Error&) { return 0; }
    return tmp.trim_spares(-1);
}

int grlgpu_destroy(grlgpu_ctx* ctx) {
    if (!ctx) return GRLGPU_ERR_ARG;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->st);
    cudaStream_t st = ctx->st;
    const bool own = ctx->own_stream;
    ctx->prof.resolve();
    if (ctx->copy_st) { cudaStreamSynchronize(ctx->copy_st); cudaStreamDestroy(ctx->copy_st); cudaEventDestroy(ctx->copy_ev); }
    for (int k = 0; k < 2; k++) {
        if (ctx->stage_buf[k]) cudaFreeHost(ctx->stage_buf[k]);
        if (ctx->stage_ev[k]) cudaEventDestroy(ctx->stage_ev[k]);
    }
    delete ctx;  // the stream was synchronised above: the pool's slabs are idle
    if (own) cudaStreamDestroy(st);
    return GRLGPU_OK;
}

static int set_text_common(grlgpu_ctx* ctx, const void* text, uint64_t n_syms, int sym_bytes, bool on_device) {
    if (!ctx || !text || n_syms == 0 || !(sym_bytes == 1 || sym_bytes == 2 || sym_bytes == 4 || sym_bytes == 8)) return GRLGPU_ERR_ARG;
    if (on_device && ((uintptr_t)text & 15)) return GRLGPU_ERR_ARG;
    return guarded(ctx, [&] {
        ctx->n = n_syms; ctx->w = sym_bytes; ctx->first = true; ctx->round = 0; ctx->done = false; ctx->have_stats = false;
        ctx->mg_n_strings = 0; ctx->mg_sl = Mg2Slices();
        if (on_device) { ctx->text_own.release(); ctx->text = text; }
        else {
            ctx->text_own.alloc(n_syms * (u64)sym_bytes + 16, ctx->st);
            GRL_CUDA(cudaMemcpyAsync(ctx->text_own.p, text, n_syms * (u64)sym_bytes, cudaMemcpyHostToDevice, ctx->st));
            GRL_CUDA(cudaStreamSynchronize(ctx->st));
            ctx->text = ctx->text_own.p;
        }
    });
}
int grlgpu_set_text(grlgpu_ctx* ctx, const void* text, uint64_t n_syms, int sym_bytes) { return set_text_common(ctx, text, n_syms, sym_bytes, false); }
int grlgpu_set_text_device(grlgpu_ctx* ctx, const void* dev_text, uint64_t n_syms, int sym_bytes) { return set_text_common(ctx, dev_text, n_syms, sym_bytes, true); }

int grlgpu_stats(grlgpu_ctx* ctx, grlgpu_stats_t* out) {
    if (!ctx || !out) return GRLGPU_ERR_ARG;
    if (!ctx->text || !ctx->first) return GRLGPU_ERR_STATE;
    int rc = guarded(ctx, [&] { ensure_stats(ctx); });
    if (rc == GRLGPU_OK) *out = ctx->stats;
    return rc;
}

int grlgpu_round(grlgpu_ctx* ctx, grlgpu_round_t* out) {
    if (!ctx || !out) return GRLGPU_ERR_ARG;
    if (!ctx->text || ctx->done) return GRLGPU_ERR_STATE;
    if (!ctx->have_stats) {
        grlgpu_stats_t s;
        int rc = grlgpu_stats(ctx, &s);
        if (rc != GRLGPU_OK) return rc;
    }
    return guarded(ctx, [&] { run_round(ctx, out); });
}

// ---- level hand-over: every way a level leaves the context (copied to the host, parked for the fetch threads) goes through
// copy_level and park ----
static __global__ void __launch_bounds__(256) narrow_u64_kernel(const u64* __restrict__ in, u64 n, u32* __restrict__ out) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (u32)in[i];
}
// the second stream of asynchronous level fetches and of the streaming ingest
static void ensure_copy_stream(grlgpu_ctx* ctx) {
    if (!ctx->copy_st) {
        GRL_CUDA(cudaStreamCreateWithFlags(&ctx->copy_st, cudaStreamNonBlocking));
        GRL_CUDA(cudaEventCreateWithFlags(&ctx->copy_ev, cudaEventDisableTiming));
    }
}
// the run lengths of `v` as 32-bit values, written on the compute stream (the caller has checked that they fit)
static DevBuf<u32> narrow_lengths(grlgpu_ctx* ctx, const LevelView& v) {
    DevBuf<u32> len32(v.n_pre, ctx->st);
    if (v.n_pre) GRL_LAUNCH("narrow_u64", v.n_pre * 12, narrow_u64_kernel, grid_for(v.n_pre, 256), 256, 0, ctx->st, v.pre_len, v.n_pre, len32.p);
    return len32;
}
// Copies the arrays of `v` whose host destination is not null, run lengths as len_bytes (4 or 8) each. Synchronous on the
// compute stream, or (async) queued on the copy stream behind the work queued on the compute stream so far: the copies then
// still read the level's arrays and the returned 32-bit lengths, and the caller parks both.
static DevBuf<u32> copy_level(grlgpu_ctx* ctx, const LevelView& v, void* rule_l, void* rule_r, u8* has_hocc, void* pre_sym, void* pre_len, int len_bytes, bool async) {
    DevBuf<u32> len32;
    if (pre_len && len_bytes == 4) len32 = narrow_lengths(ctx, v);
    cudaStream_t cs = ctx->st;
    if (async) {
        ensure_copy_stream(ctx);
        GRL_CUDA(cudaEventRecord(ctx->copy_ev, ctx->st));
        GRL_CUDA(cudaStreamWaitEvent(ctx->copy_st, ctx->copy_ev, 0));
        cs = ctx->copy_st;
    }
    const u64 sb = (u64)v.sym_bytes;
    const void* lens = len32.p ? (const void*)len32.p : (const void*)v.pre_len;
    struct Copy { void* dst; const void* src; u64 bytes; };
    for (const Copy& c : {Copy{rule_l, v.rule_l, v.tot * sb}, Copy{rule_r, v.rule_r, v.tot * sb}, Copy{has_hocc, v.has_hocc, v.tot}, Copy{pre_sym, v.pre_sym, v.n_pre * sb},
                          Copy{pre_len, lens, v.n_pre * (u64)len_bytes}})
        if (c.dst) GRL_CUDA(cudaMemcpyAsync(c.dst, c.src, c.bytes, cudaMemcpyDeviceToHost, cs));
    if (!async) GRL_CUDA(cudaStreamSynchronize(ctx->st));
    return len32;
}
// Keeps a level's arrays out of the pool until grlgpu_fetch_wait. len32: the 32-bit run lengths the host takes instead of the
// 64-bit ones; those then go back to the pool at once, since their only reader, narrow_u64, runs on the compute stream before
// the pool can hand the memory out again.
static void park(grlgpu_ctx* ctx, DevLevel&& L, DevBuf<u32>&& len32) {
    if (len32.p) L.pre_len.release();
    ctx->parked.push_back({std::move(L), std::move(len32)});
}

int grlgpu_fetch_level(grlgpu_ctx* ctx, void* rule_l, void* rule_r, uint8_t* has_hocc, void* pre_sym, uint64_t* pre_len) {
    if (!ctx) return GRLGPU_ERR_ARG;
    if (ctx->round == 0 || !ctx->lvl.present()) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] { copy_level(ctx, view_of(ctx->lvl), rule_l, rule_r, has_hocc, pre_sym, pre_len, 8, false); });
}

// Same as grlgpu_fetch_level / _async with 32-bit run lengths (the run lengths of a level sum to at most n_in + parse_len,
// so this applies whenever that is < 2^32): 4 bytes less per preliminary-BWT run over PCIe.
int grlgpu_fetch_level32(grlgpu_ctx* ctx, void* rule_l, void* rule_r, uint8_t* has_hocc, void* pre_sym, uint32_t* pre_len32, int async) {
    if (!ctx) return GRLGPU_ERR_ARG;
    if (ctx->round == 0 || !ctx->lvl.present()) return GRLGPU_ERR_STATE;
    if (ctx->lvl_n_in >= (1ull << 32)) return GRLGPU_ERR_LIMIT;
    return guarded(ctx, [&] {
        DevBuf<u32> len32 = copy_level(ctx, view_of(ctx->lvl), rule_l, rule_r, has_hocc, pre_sym, pre_len32, 4, async != 0);
        if (async) park(ctx, std::move(ctx->lvl), std::move(len32));
    });
}

int grlgpu_fetch_level_async(grlgpu_ctx* ctx, void* rule_l, void* rule_r, uint8_t* has_hocc, void* pre_sym, uint64_t* pre_len) {
    if (!ctx) return GRLGPU_ERR_ARG;
    if (ctx->round == 0 || !ctx->lvl.present()) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] {
        DevBuf<u32> len32 = copy_level(ctx, view_of(ctx->lvl), rule_l, rule_r, has_hocc, pre_sym, pre_len, 8, true);
        park(ctx, std::move(ctx->lvl), std::move(len32));
    });
}

int grlgpu_level_checksum(grlgpu_ctx* ctx, uint64_t* out4) {
    if (!ctx || !out4) return GRLGPU_ERR_ARG;
    if (ctx->round == 0 || !ctx->lvl.present()) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] { level_checksum(ctx->st, view_of(ctx->lvl), (u64*)out4); });
}

// ---- streaming ingest: the caller fills pinned staging buffers (e.g. read() straight from the input file), the copies to the
// device run on the copy stream while the caller fills the other buffer ----
int grlgpu_text_begin(grlgpu_ctx* ctx, uint64_t n_syms, int sym_bytes, uint64_t stage_bytes) {
    if (!ctx || n_syms == 0 || !(sym_bytes == 1 || sym_bytes == 2 || sym_bytes == 4 || sym_bytes == 8)) return GRLGPU_ERR_ARG;
    return guarded(ctx, [&] {
        ensure_copy_stream(ctx);
        const u64 cap = std::max<u64>(1ull << 20, (stage_bytes ? stage_bytes : (16ull << 20)) / 4096 * 4096);
        if (cap != ctx->stage_cap) {
            for (int k = 0; k < 2; k++) {
                if (ctx->stage_buf[k]) { GRL_CUDA(cudaFreeHost(ctx->stage_buf[k])); ctx->stage_buf[k] = nullptr; }
                GRL_CUDA(cudaHostAlloc((void**)&ctx->stage_buf[k], cap, cudaHostAllocDefault));
                if (!ctx->stage_ev[k]) GRL_CUDA(cudaEventCreateWithFlags(&ctx->stage_ev[k], cudaEventDisableTiming));
            }
            ctx->stage_cap = cap;
        }
        ctx->n = n_syms; ctx->w = sym_bytes; ctx->first = true; ctx->round = 0; ctx->done = false; ctx->have_stats = false;
        ctx->mg_n_strings = 0; ctx->mg_sl = Mg2Slices();
        ctx->ingest_bytes = n_syms * (u64)sym_bytes;
        ctx->ingest_off = 0;
        ctx->stage_cur = 0;
        ctx->text_own.alloc(ctx->ingest_bytes + 16, ctx->st);
        ctx->text = ctx->text_own.p;
        GRL_CUDA(cudaStreamSynchronize(ctx->st));  // the block may have been in use by earlier work of the compute stream
        ctx->ingesting = true;
    });
}
int grlgpu_text_stage(grlgpu_ctx* ctx, void** buf, uint64_t* cap) {
    if (!ctx || !buf || !cap) return GRLGPU_ERR_ARG;
    if (!ctx->ingesting) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] {
        GRL_CUDA(cudaEventSynchronize(ctx->stage_ev[ctx->stage_cur]));  // the previous copy out of this buffer is done
        *buf = ctx->stage_buf[ctx->stage_cur];
        *cap = std::min<u64>(ctx->stage_cap, ctx->ingest_bytes - ctx->ingest_off);
    });
}
int grlgpu_text_commit(grlgpu_ctx* ctx, uint64_t bytes) {
    if (!ctx) return GRLGPU_ERR_ARG;
    if (!ctx->ingesting || bytes > ctx->stage_cap || ctx->ingest_off + bytes > ctx->ingest_bytes) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] {
        const int k = ctx->stage_cur;
        GRL_CUDA(cudaMemcpyAsync(ctx->text_own.p + ctx->ingest_off, ctx->stage_buf[k], bytes, cudaMemcpyHostToDevice, ctx->copy_st));
        GRL_CUDA(cudaEventRecord(ctx->stage_ev[k], ctx->copy_st));
        ctx->ingest_off += bytes;
        ctx->stage_cur ^= 1;
    });
}
int grlgpu_text_end(grlgpu_ctx* ctx) {
    if (!ctx) return GRLGPU_ERR_ARG;
    if (!ctx->ingesting) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] {
        ctx->ingesting = false;
        if (ctx->ingest_off != ctx->ingest_bytes) throw Error(GRLGPU_ERR_STATE, "text ingest ended before every byte was committed");
        GRL_CUDA(cudaStreamSynchronize(ctx->copy_st));
    });
}

// ---- level hand-over for host-side fetch threads: the level's device arrays are parked (kept alive, not returned to the pool)
// and their addresses given out; any host thread may then copy them with grlgpu_copy_to_host while this context computes the
// next round. grlgpu_fetch_wait releases them. Works for the level of grlgpu_round and for the slice of grlgpu_mg_round. ----
int grlgpu_level_park(grlgpu_ctx* ctx, int len_bytes, grlgpu_level_ptrs_t* out) {
    if (!ctx || !out || !(len_bytes == 4 || len_bytes == 8)) return GRLGPU_ERR_ARG;
    const bool mg = ctx->mg_sl.valid;
    if (!mg && (ctx->round == 0 || !ctx->lvl.present())) return GRLGPU_ERR_STATE;
    if (!mg && len_bytes == 4 && ctx->lvl_n_in >= (1ull << 32)) return GRLGPU_ERR_LIMIT;
    return guarded(ctx, [&] {
        memset(out, 0, sizeof(*out));
        const LevelView v = mg ? ctx->mg_sl.view() : view_of(ctx->lvl);
        DevBuf<u32> len32;
        if (len_bytes == 4) len32 = narrow_lengths(ctx, v);
        GRL_CUDA(cudaStreamSynchronize(ctx->st));
        out->device = ctx->device;
        out->sym_bytes = (uint32_t)v.sym_bytes; out->len_bytes = (uint32_t)len_bytes; out->tot = v.tot; out->n_pre = v.n_pre;
        out->rule_l = v.rule_l; out->rule_r = v.rule_r; out->has_hocc = v.has_hocc; out->pre_sym = v.pre_sym;
        out->pre_len = len32.p ? (const void*)len32.p : (const void*)v.pre_len;
        park(ctx, std::move(mg ? ctx->mg_sl.lvl : ctx->lvl), std::move(len32));
        ctx->mg_sl.valid = false;
    });
}
// blocking device -> host copy on a stream private to the calling thread; thread-safe, needs no context
int grlgpu_copy_to_host(int device, void* dst, const void* dev_src, uint64_t bytes) {
    if (bytes == 0) return GRLGPU_OK;
    if (!dst || !dev_src) return GRLGPU_ERR_ARG;
    static thread_local cudaStream_t s[64] = {nullptr};
    if (device < 0 || device >= 64) return GRLGPU_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) return GRLGPU_ERR_CUDA;
    if (!s[device] && cudaStreamCreateWithFlags(&s[device], cudaStreamNonBlocking) != cudaSuccess) return GRLGPU_ERR_CUDA;
    if (cudaMemcpyAsync(dst, dev_src, bytes, cudaMemcpyDeviceToHost, s[device]) != cudaSuccess) return GRLGPU_ERR_CUDA;
    return cudaStreamSynchronize(s[device]) == cudaSuccess ? GRLGPU_OK : GRLGPU_ERR_CUDA;
}

int grlgpu_fetch_wait(grlgpu_ctx* ctx) {
    if (!ctx) return GRLGPU_ERR_ARG;
    return guarded(ctx, [&] {
        if (ctx->copy_st) GRL_CUDA(cudaStreamSynchronize(ctx->copy_st));
        ctx->parked.clear();
    });
}

int grlgpu_fetch_parse(grlgpu_ctx* ctx, void* dst) {
    if (!ctx || !dst) return GRLGPU_ERR_ARG;
    if (ctx->round == 0) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] {
        GRL_CUDA(cudaMemcpyAsync(dst, ctx->text, ctx->n * (u64)ctx->w, cudaMemcpyDeviceToHost, ctx->st));
        GRL_CUDA(cudaStreamSynchronize(ctx->st));
    });
}

int grlgpu_fetch_str_ptrs(grlgpu_ctx* ctx, uint64_t* dst) {
    if (!ctx || !dst) return GRLGPU_ERR_ARG;
    if (ctx->round == 0) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] {
        const u64 n_words = div_up(ctx->n, 32);
        DevBuf<u32> sb(n_words, ctx->st);
        GRL_LAUNCH("next_start_bits", 0, next_start_bits_kernel, grid_for(n_words, 256), 256, 0, ctx->st, ctx->end_bits.p, ctx->n, sb.p);
        BitmapCompactor bc;
        const u64 ns = bc.count(sb.p, ctx->n, ctx->st);
        if (ns != ctx->n_strings) throw Error(GRLGPU_ERR_STATE, "string count changed between rounds");
        DevBuf<u64> ptrs(ns + 1, ctx->st);
        bc.write<u64>(nullptr, ptrs.p);
        GRL_CUDA(cudaMemcpyAsync(dst, ptrs.p, ns * 8, cudaMemcpyDeviceToHost, ctx->st));
        GRL_CUDA(cudaStreamSynchronize(ctx->st));
        dst[ns] = ctx->n;
    });
}

int grlgpu_fetch_dictionary(grlgpu_ctx* ctx, uint64_t* syms, uint64_t* lens, uint64_t* freqs, uint64_t* metas) {
    if (!ctx) return GRLGPU_ERR_ARG;
    if (ctx->round == 0 || !(ctx->flags & GRLGPU_FLAG_KEEP_DICT) || !ctx->kd_order.p) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] {
        const u64 d = ctx->kd_d, nE = ctx->kd_nE, nS = ctx->kd_nS;
        std::vector<u32> order(nS), phr_of(nE), off(d + 1), len(d);
        std::vector<u64> freq(d), meta(d);
        std::vector<u8> Draw(nE * (u64)ctx->lvl.sym_bytes);
        GRL_CUDA(cudaMemcpy(order.data(), ctx->kd_order.p, nS * 4, cudaMemcpyDeviceToHost));
        GRL_CUDA(cudaMemcpy(phr_of.data(), ctx->kd_phr_of.p, nE * 4, cudaMemcpyDeviceToHost));
        GRL_CUDA(cudaMemcpy(off.data(), ctx->kd_off.p, (d + 1) * 4, cudaMemcpyDeviceToHost));
        GRL_CUDA(cudaMemcpy(len.data(), ctx->kd_len.p, d * 4, cudaMemcpyDeviceToHost));
        GRL_CUDA(cudaMemcpy(freq.data(), ctx->kd_freq.p, d * 8, cudaMemcpyDeviceToHost));
        GRL_CUDA(cudaMemcpy(meta.data(), ctx->kd_meta.p, d * 8, cudaMemcpyDeviceToHost));
        GRL_CUDA(cudaMemcpy(Draw.data(), ctx->kd_D.p, Draw.size(), cudaMemcpyDeviceToHost));
        u64 k = 0, so = 0;
        for (u64 i = 0; i < nS; i++) {  // full-phrase entries in suffix order = phrases in A.2 order
            const u32 e = order[i], ph = phr_of[e];
            if (e != off[ph]) continue;
            if (lens) lens[k] = len[ph];
            if (freqs) freqs[k] = freq[ph];
            if (metas) metas[k] = meta[ph];
            if (syms)
                for (u32 t = 0; t < len[ph]; t++)
                    syms[so + t] = ctx->lvl.sym_bytes == 4 ? ((const u32*)Draw.data())[e + t] : ((const u64*)Draw.data())[e + t];
            so += len[ph];
            k++;
        }
    });
}

int grlgpu_histogram(grlgpu_ctx* ctx, uint64_t* hist256) {
    if (!ctx || !hist256) return GRLGPU_ERR_ARG;
    if (!ctx->have_stats) return GRLGPU_ERR_STATE;
    memcpy(hist256, ctx->hist, sizeof(ctx->hist));
    return GRLGPU_OK;
}

// ---- exchange layer + multi-GPU rounds (comm.hpp, mg2.cuh) ----
int grlgpu_nccl_unique_id(void* id128) {
    if (!id128) return GRLGPU_ERR_ARG;
    return guarded(nullptr, [&] {
        NcclApi& api = NcclApi::get();
        ncclUniqueId id;
        GRL_NCCL(api.GetUniqueId(&id));
        memcpy(id128, &id, sizeof(id));
    });
}
int grlgpu_comm_create_nccl(grlgpu_comm** comm, const void* id128, int rank, int world, int device) {
    if (!comm || !id128 || world < 1 || world > 31 || rank < 0 || rank >= world) return GRLGPU_ERR_ARG;
    *comm = nullptr;
    return guarded(nullptr, [&] {
        std::unique_ptr<grlgpu_comm> h(new grlgpu_comm());
        h->c.reset(new NcclComm(id128, rank, world, device));
        *comm = h.release();
    });
}
int grlgpu_comm_create_ipc(grlgpu_comm** comm, const char* session, int rank, int world, int device) {
    if (!comm || !session || session[0] != '/' || world < 1 || world > 31 || rank < 0 || rank >= world) return GRLGPU_ERR_ARG;
    *comm = nullptr;
    return guarded(nullptr, [&] {
        std::unique_ptr<grlgpu_comm> h(new grlgpu_comm());
        h->c.reset(new IpcComm(session, rank, world, device));
        *comm = h.release();
    });
}
// CPU self-test of the shared-memory rendezvous (no GPU involved): `rounds` barriers and small all-gathers of payloads of varying size
// between `world` processes; returns GRLGPU_OK when every gathered byte is what its rank wrote
int grlgpu_selftest_ipc_rendezvous(const char* session, int rank, int world, int rounds) {
    if (!session || session[0] != '/' || world < 1 || world > 31 || rank < 0 || rank >= world || rounds < 1) return GRLGPU_ERR_ARG;
    return guarded(nullptr, [&] {
        IpcComm cm(session, rank, world, 0, /*with_cuda=*/false);
        for (int r = 0; r < rounds; r++) {
            const size_t n = (size_t)1 + ((size_t)r * 7919u) % 100000u;  // up to ~800 KB per rank: several 64 KB pieces
            std::vector<u64> mine(n), all(n * (size_t)world);
            for (size_t i = 0; i < n; i++) mine[i] = ((u64)rank << 48) ^ ((u64)r << 24) ^ (u64)i;
            cm.all_gather_host(mine.data(), n * sizeof(u64), all.data(), nullptr);
            for (int p = 0; p < world; p++)
                for (size_t i = 0; i < n; i++)
                    if (all[(size_t)p * n + i] != (((u64)p << 48) ^ ((u64)r << 24) ^ (u64)i)) { cm.abort_group(); throw Error(GRLGPU_ERR_STATE, "rendezvous self-test: wrong byte gathered"); }
            cm.barrier();
        }
    });
}
int grlgpu_local_group_create(grlgpu_local_group** group, int world) {
    if (!group || world < 1 || world > 31) return GRLGPU_ERR_ARG;
    *group = new grlgpu_local_group(world);
    return GRLGPU_OK;
}
int grlgpu_local_group_abort(grlgpu_local_group* group) {
    if (!group) return GRLGPU_ERR_ARG;
    group->g.abort();
    return GRLGPU_OK;
}
int grlgpu_local_group_destroy(grlgpu_local_group* group) {
    delete group;
    return GRLGPU_OK;
}
int grlgpu_comm_create_local(grlgpu_comm** comm, grlgpu_local_group* group, int rank, int device) {
    if (!comm || !group || rank < 0 || rank >= group->g.world) return GRLGPU_ERR_ARG;
    std::unique_ptr<grlgpu_comm> h(new grlgpu_comm());
    h->c.reset(new LocalComm(&group->g, rank, device));
    *comm = h.release();
    return GRLGPU_OK;
}
int grlgpu_comm_destroy(grlgpu_comm* comm) {
    if (comm) cudaSetDevice(comm->c->device);
    delete comm;
    return GRLGPU_OK;
}
int grlgpu_comm_times(const grlgpu_comm* comm, double* ms_bulk, double* ms_small) {
    if (!comm) return GRLGPU_ERR_ARG;
    if (ms_bulk) *ms_bulk = comm->c->ms_bulk;
    if (ms_small) *ms_small = comm->c->ms_small;
    return GRLGPU_OK;
}
int grlgpu_comm_info(const grlgpu_comm* comm, uint64_t* bytes_sent, uint64_t* n_bulk, uint64_t* n_small, char* kind, int kind_cap) {
    if (!comm) return GRLGPU_ERR_ARG;
    if (bytes_sent) *bytes_sent = comm->c->bytes_sent;
    if (n_bulk) *n_bulk = comm->c->n_bulk;
    if (n_small) *n_small = comm->c->n_small;
    if (kind && kind_cap > 0) snprintf(kind, (size_t)kind_cap, "%s", comm->c->kind());
    return GRLGPU_OK;
}
int grlgpu_can_peer(int device_a, int device_b) {
    if (device_a == device_b) return 1;
    int ab = 0, ba = 0;
    if (cudaDeviceCanAccessPeer(&ab, device_a, device_b) != cudaSuccess || cudaDeviceCanAccessPeer(&ba, device_b, device_a) != cudaSuccess) { cudaGetLastError(); return 0; }
    return ab && ba;
}
int grlgpu_set_peers(grlgpu_ctx* ctx, const int* devices, int n_devices) {
    if (!ctx || (n_devices > 0 && !devices) || n_devices < 0) return GRLGPU_ERR_ARG;
    return guarded(ctx, [&] {
        // runtime peer copies (cudaMemcpyPeerAsync) are staged through host memory unless peer access is enabled between the two
        // devices' contexts; with it they are direct NVLink DMA. Enabled once per pair and process ("already enabled" is fine).
        for (int i = 0; i < n_devices; i++) {
            if (devices[i] == ctx->device || !grlgpu_can_peer(ctx->device, devices[i])) continue;
            const cudaError_t e = cudaDeviceEnablePeerAccess(devices[i], 0);
            if (e != cudaSuccess) cudaGetLastError();  // cudaErrorPeerAccessAlreadyEnabled, or unsupported: the copies then take the staged path
        }
        ctx->pool.set_peers(std::vector<int>(devices, devices + n_devices));
    });
}

int grlgpu_mg_stats(grlgpu_ctx* ctx, grlgpu_comm* comm, grlgpu_stats_t* out) {
    if (!ctx || !comm || !out) return GRLGPU_ERR_ARG;
    if (!ctx->text || !ctx->first) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] {
        Comm& cm = *comm->c;
        // local statistics first; a rank whose shard is ill formed reports it so that every rank fails together
        std::vector<u64> mine(7 + 256, 0);
        int rc = GRLGPU_OK;
        try { ensure_stats(ctx); }
        catch (const Error& e) { rc = e.code; ctx->last_error = e.what(); cudaGetLastError(); }
        mine[0] = (u64)(int64_t)rc;
        if (rc == GRLGPU_OK) {
            const grlgpu_stats_t& s = ctx->stats;
            mine[1] = s.n_syms; mine[2] = s.n_strings; mine[3] = s.longest_string; mine[4] = s.min_sym; mine[5] = s.max_sym; mine[6] = s.sep_sym;
            memcpy(mine.data() + 7, ctx->hist, sizeof(ctx->hist));
        }
        const std::vector<u64> all = mg2_gather(cm, mine, ctx->st);
        grlgpu_stats_t g{};
        g.min_sym = ~0ULL;
        u64 hist[256] = {0};
        for (int p = 0; p < cm.world; p++) {
            const u64* row = all.data() + (size_t)p * mine.size();
            if ((int)(int64_t)row[0] != GRLGPU_OK) throw Error((int)(int64_t)row[0], "rank " + std::to_string(p) + ": " + grlgpu_strerror((int)(int64_t)row[0]));
            g.n_syms += row[1]; g.n_strings += row[2];
            g.longest_string = std::max<u64>(g.longest_string, row[3]);
            g.min_sym = std::min<u64>(g.min_sym, row[4]);
            g.max_sym = std::max<u64>(g.max_sym, row[5]);
            if (p == 0) g.sep_sym = row[6];
            else if (row[6] != g.sep_sym) throw Error(GRLGPU_ERR_ILL_FORMED, "the collection is ill formed: the shards end in different symbols");
            for (int k = 0; k < 256; k++) hist[k] += row[7 + k];
        }
        if (g.sep_sym != g.min_sym) throw Error(GRLGPU_ERR_ILL_FORMED, "the collection is ill formed: the last symbol is not the smallest symbol");
        g.max_sym_freq = g.n_syms;  // utils.cpp:117
        if (ctx->w == 1) {          // utils.cpp:161-175 on the global histogram
            u64 mx = 0;
            for (int k = 0; k < 256; k++) mx = std::max(mx, hist[k]);
            g.max_sym_freq = mx;
        }
        ctx->alphabet = g.max_sym + 1;  // exact_par_phase.cpp:316, over the whole collection
        ctx->mg_n_strings = g.n_strings;
        *out = g;
    });
}

int grlgpu_mg_round(grlgpu_ctx* ctx, grlgpu_comm* comm, grlgpu_round_t* out) {
    if (!ctx || !comm || !out) return GRLGPU_ERR_ARG;
    if (!ctx->text || ctx->done || !ctx->have_stats || !ctx->mg_n_strings) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] {
        Comm& cm = *comm->c;
        struct AbortOnThrow {  // a rank that fails inside the round must not leave its peers waiting in an exchange
            Comm& cm; bool armed = true;
            ~AbortOnThrow() { if (armed) cm.abort_group(); }
        } guard{cm};
        if (ctx->first) switch (ctx->w) {
            case 1: mg2_round_t<u8, true>(ctx, cm, out); break;
            case 2: mg2_round_t<u16, true>(ctx, cm, out); break;
            case 4: mg2_round_t<u32, true>(ctx, cm, out); break;
            default: mg2_round_t<u64, true>(ctx, cm, out); break;
        } else switch (ctx->w) {
            case 1: mg2_round_t<u8, false>(ctx, cm, out); break;
            case 2: mg2_round_t<u16, false>(ctx, cm, out); break;
            case 4: mg2_round_t<u32, false>(ctx, cm, out); break;
            default: mg2_round_t<u64, false>(ctx, cm, out); break;
        }
        guard.armed = false;
    });
}

int grlgpu_mg_slice_info(grlgpu_ctx* ctx, grlgpu_slice_t* out) {
    if (!ctx || !out) return GRLGPU_ERR_ARG;
    if (!ctx->mg_n_strings || ctx->round == 0) return GRLGPU_ERR_STATE;
    const Mg2Slices& S = ctx->mg_sl;
    out->rank_base = S.rank_base; out->tot_local = S.lvl.tot; out->pre_first = S.pre_first; out->n_pre_local = S.lvl.n_pre - S.pre_drop;
    out->exchange_bytes = ctx->mg_exchange_bytes; out->sym_bytes = (uint32_t)S.lvl.sym_bytes; out->reserved = 0;
    out->n_in_local = ctx->mg_n_in_local; out->parse_len_local = ctx->mg_parse_len_local;
    return GRLGPU_OK;
}

int grlgpu_mg_fetch_slice(grlgpu_ctx* ctx, void* rule_l, void* rule_r, uint8_t* has_hocc, void* pre_sym, void* pre_len, int len_bytes, int async) {
    if (!ctx || !(len_bytes == 4 || len_bytes == 8)) return GRLGPU_ERR_ARG;
    if (!ctx->mg_sl.valid) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] {
        Mg2Slices& S = ctx->mg_sl;
        DevBuf<u32> len32 = copy_level(ctx, S.view(), rule_l, rule_r, has_hocc, pre_sym, pre_len, len_bytes, async != 0);
        if (async) {  // the slice cannot be fetched again
            park(ctx, std::move(S.lvl), std::move(len32));
            S.valid = false;
        }
    });
}

int grlgpu_mg_slice_checksum(grlgpu_ctx* ctx, uint64_t* out4) {
    if (!ctx || !out4) return GRLGPU_ERR_ARG;
    if (!ctx->mg_sl.valid) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] { level_checksum(ctx->st, ctx->mg_sl.view(), (u64*)out4); });
}

// ---- induction phase on the device (induce.cuh) ----
int grlgpu_keep_level(grlgpu_ctx* ctx) {
    if (!ctx) return GRLGPU_ERR_ARG;
    if (ctx->round == 0 || !ctx->lvl.present()) return GRLGPU_ERR_STATE;
    if (ctx->lvl.sym_bytes != 4) return GRLGPU_ERR_LIMIT;
    return guarded(ctx, [&] { ctx->kept.push_back({ctx->lvl_alphabet, std::move(ctx->lvl)}); });
}
int grlgpu_level_adopt(grlgpu_ctx* ctx, uint64_t alphabet, uint64_t tot, uint64_t n_pre, grlgpu_level_ptrs_t* out) {
    if (!ctx || !out) return GRLGPU_ERR_ARG;
    return guarded(ctx, [&] {
        DevLevel L;
        L.tot = tot; L.n_pre = n_pre;
        L.rule_l.alloc(tot * 4, ctx->st); L.rule_r.alloc(tot * 4, ctx->st); L.has_hocc.alloc(tot, ctx->st);
        L.pre_sym.alloc(n_pre * 4, ctx->st); L.pre_len.alloc(n_pre, ctx->st);
        memset(out, 0, sizeof(*out));
        out->rule_l = L.rule_l.p; out->rule_r = L.rule_r.p; out->has_hocc = L.has_hocc.p; out->pre_sym = L.pre_sym.p; out->pre_len = L.pre_len.p;
        out->tot = tot; out->n_pre = n_pre; out->sym_bytes = 4; out->len_bytes = 8; out->device = ctx->device;
        ctx->kept.push_back({alphabet, std::move(L)});
        GRL_CUDA(cudaStreamSynchronize(ctx->st));
    });
}
int grlgpu_copy_dev(int dst_device, void* dst, int src_device, const void* src, uint64_t bytes) {
    if (bytes == 0) return GRLGPU_OK;
    if (!dst || !src || dst_device < 0 || dst_device >= 64) return GRLGPU_ERR_ARG;
    // cudaMemcpyPeer / device-to-device cudaMemcpy return before the copy has finished: use a stream private to the calling
    // thread and wait for it, so that the caller may release the source as soon as this returns
    static thread_local cudaStream_t s[64] = {nullptr};
    if (cudaSetDevice(dst_device) != cudaSuccess) return GRLGPU_ERR_CUDA;
    if (!s[dst_device] && cudaStreamCreateWithFlags(&s[dst_device], cudaStreamNonBlocking) != cudaSuccess) return GRLGPU_ERR_CUDA;
    const cudaError_t e = dst_device == src_device ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s[dst_device])
                                                   : cudaMemcpyPeerAsync(dst, dst_device, src, src_device, bytes, s[dst_device]);
    if (e != cudaSuccess) return GRLGPU_ERR_CUDA;
    return cudaStreamSynchronize(s[dst_device]) == cudaSuccess ? GRLGPU_OK : GRLGPU_ERR_CUDA;
}
int grlgpu_device_of(const grlgpu_ctx* ctx) { return ctx ? ctx->device : -1; }
int grlgpu_kept_levels(const grlgpu_ctx* ctx) { return ctx ? (int)ctx->kept.size() : 0; }
int grlgpu_fetch_kept_level(grlgpu_ctx* ctx, int level, uint64_t* alphabet, uint64_t* tot, uint64_t* n_pre, void* rule_l, void* rule_r, uint8_t* has_hocc, void* pre_sym,
                            uint64_t* pre_len) {
    if (!ctx || level < 0 || (size_t)level >= ctx->kept.size()) return GRLGPU_ERR_ARG;
    return guarded(ctx, [&] {
        const IndLevel& K = ctx->kept[(size_t)level];
        if (alphabet) *alphabet = K.alphabet;
        if (tot) *tot = K.lvl.tot;
        if (n_pre) *n_pre = K.lvl.n_pre;
        copy_level(ctx, view_of(K.lvl), rule_l, rule_r, has_hocc, pre_sym, pre_len, 8, false);
    });
}
int grlgpu_drop_kept(grlgpu_ctx* ctx) {
    if (!ctx) return GRLGPU_ERR_ARG;
    return guarded(ctx, [&] { ctx->kept.clear(); ctx->bwt_dev = IndBwt(); ctx->bwt_ready = false; });
}
int grlgpu_induce(grlgpu_ctx* ctx, const void* final_parse, uint64_t n_strings, int cell_bytes, uint64_t n_syms_total, uint64_t* n_runs) {
    if (!ctx || !n_runs || !(cell_bytes == 1 || cell_bytes == 2 || cell_bytes == 4 || cell_bytes == 8)) return GRLGPU_ERR_ARG;
    if (ctx->kept.empty()) return GRLGPU_ERR_STATE;
    if (n_syms_total >= 0xfffffff0ull || n_strings >= 0xfffffff0ull) return GRLGPU_ERR_LIMIT;  // 32-bit offsets on the device
    return guarded(ctx, [&] {
        cudaStream_t st = ctx->st;
        const bool trace = getenv("GRLGPU_TRACE") != nullptr;
        ctx->bwt_ready = false;
        const u32 n = (u32)n_strings;
        IndBwt bwt;
        {   // deepest level: the final parse in string order (host buffer, or this context's own current parse)
            DevBuf<u8> fp;
            const void* dparse = ctx->text;
            if (final_parse) {
                fp.alloc(n_strings * (u64)cell_bytes + 16, st);
                GRL_CUDA(cudaMemcpyAsync(fp.p, final_parse, n_strings * (u64)cell_bytes, cudaMemcpyHostToDevice, st));
                dparse = fp.p;
            } else if (!ctx->done || ctx->n != n_strings || ctx->w != cell_bytes) throw Error(GRLGPU_ERR_STATE, "no final parse in the context");
            DevBuf<u32> sym(n, st);
            switch (cell_bytes) {
                case 1: GRL_LAUNCH("ind_parse_syms", n * 5, (ind_parse_syms_kernel<u8>), grid_for(n, 256), 256, 0, st, (const u8*)dparse, n, sym.p); break;
                case 2: GRL_LAUNCH("ind_parse_syms", n * 6, (ind_parse_syms_kernel<u16>), grid_for(n, 256), 256, 0, st, (const u16*)dparse, n, sym.p); break;
                case 4: GRL_LAUNCH("ind_parse_syms", n * 8, (ind_parse_syms_kernel<u32>), grid_for(n, 256), 256, 0, st, (const u32*)dparse, n, sym.p); break;
                default: GRL_LAUNCH("ind_parse_syms", n * 12, (ind_parse_syms_kernel<u64>), grid_for(n, 256), 256, 0, st, (const u64*)dparse, n, sym.p); break;
            }
            ind_maximal_runs(sym.p, nullptr, n, n, bwt, st);
        }
        // (the kept levels are only dropped once the whole induction has succeeded: after a failure the caller can still fetch them)
        for (size_t lv = ctx->kept.size(); lv-- > 0;) {
            Timer t(st);
            t.start();
            ind_level_step(bwt, ctx->kept[lv], st, trace);
            t.stop();
            if (trace) fprintf(stderr, "[grlgpu] induction: level %zu took %.2f ms\n", lv, t.ms());
        }
        ctx->kept.clear();
        if ((u64)bwt.n_syms != n_syms_total) throw Error(GRLGPU_ERR_STATE, "induction: the level-0 BWT does not have one symbol per input symbol");
        *n_runs = bwt.n_runs;
        ctx->bwt_dev = std::move(bwt);
        ctx->bwt_ready = true;
    });
}
int grlgpu_bwt_ptrs(grlgpu_ctx* ctx, const uint32_t** d_syms, const uint32_t** d_lens, uint64_t* n_runs) {
    if (!ctx || !d_syms || !d_lens || !n_runs) return GRLGPU_ERR_ARG;
    if (!ctx->bwt_ready) return GRLGPU_ERR_STATE;
    *d_syms = ctx->bwt_dev.sym.p; *d_lens = ctx->bwt_dev.len.p; *n_runs = ctx->bwt_dev.n_runs;
    return GRLGPU_OK;
}
int grlgpu_fetch_bwt(grlgpu_ctx* ctx, uint32_t* syms, uint32_t* lens) {
    if (!ctx || !syms || !lens) return GRLGPU_ERR_ARG;
    if (!ctx->bwt_ready) return GRLGPU_ERR_STATE;
    return guarded(ctx, [&] {
        GRL_CUDA(cudaMemcpyAsync(syms, ctx->bwt_dev.sym.p, (u64)ctx->bwt_dev.n_runs * 4, cudaMemcpyDeviceToHost, ctx->st));
        GRL_CUDA(cudaMemcpyAsync(lens, ctx->bwt_dev.len.p, (u64)ctx->bwt_dev.n_runs * 4, cudaMemcpyDeviceToHost, ctx->st));
        GRL_CUDA(cudaStreamSynchronize(ctx->st));
    });
}

int grlgpu_fetch_bwt_packed(grlgpu_ctx* ctx, int sb, int fb, void* out, uint64_t cap_bytes, uint64_t* n_bytes) {
    if (!ctx || !out || sb < 1 || sb > 8 || fb < 1 || fb > 8) return GRLGPU_ERR_ARG;
    if (!ctx->bwt_ready) return GRLGPU_ERR_STATE;
    const u64 n = ctx->bwt_dev.n_runs, rec = (u64)(sb + fb), need = 16 + n * rec;
    if (n_bytes) *n_bytes = need;
    if (cap_bytes < need) return GRLGPU_ERR_ARG;
    return guarded(ctx, [&] {
        cudaStream_t st = ctx->st;
        // [sb u64][fb u64][records]: the image of the .rl_bwt file. The records are packed piece by piece into two device buffers, so a
        // piece travels to the host while the next one is being packed
        const u64 hdr[2] = {(u64)sb, (u64)fb};
        memcpy(out, hdr, 16);
        if (n == 0) return;
        ensure_copy_stream(ctx);
        const u64 piece = std::min<u64>(n, (u64)IND_PACK_RUNS * 32768);  // 32 M runs
        DevBuf<u8> buf0(piece * rec, st), buf1(piece * rec, st);
        DevBuf<u32> err(1, st);
        err.zero();
        cudaEvent_t packed[2], copied[2];
        for (int k = 0; k < 2; k++) { GRL_CUDA(cudaEventCreateWithFlags(&packed[k], cudaEventDisableTiming)); GRL_CUDA(cudaEventCreateWithFlags(&copied[k], cudaEventDisableTiming)); }
        int k = 0;
        bool used[2] = {false, false};
        for (u64 first = 0; first < n; first += piece, k ^= 1) {
            const u64 m = std::min(piece, n - first);
            u8* d = k ? buf1.p : buf0.p;
            if (used[k]) GRL_CUDA(cudaStreamWaitEvent(st, copied[k], 0));  // the copy that last read this buffer
            GRL_LAUNCH("ind_pack_records", m * (8 + rec), ind_pack_records_kernel, (unsigned)div_up(m, IND_PACK_RUNS), 256, (size_t)IND_PACK_RUNS * rec, st, ctx->bwt_dev.sym.p,
                       ctx->bwt_dev.len.p, first, m, sb, fb, d, err.p);
            GRL_CUDA(cudaEventRecord(packed[k], st));
            GRL_CUDA(cudaStreamWaitEvent(ctx->copy_st, packed[k], 0));
            GRL_CUDA(cudaMemcpyAsync((u8*)out + 16 + first * rec, d, m * rec, cudaMemcpyDeviceToHost, ctx->copy_st));
            GRL_CUDA(cudaEventRecord(copied[k], ctx->copy_st));
            used[k] = true;
        }
        GRL_CUDA(cudaStreamSynchronize(ctx->copy_st));
        GRL_CUDA(cudaStreamSynchronize(st));
        for (int q = 0; q < 2; q++) { cudaEventDestroy(packed[q]); cudaEventDestroy(copied[q]); }
        if (d2h_scalar(err.p, st)) throw Error(GRLGPU_ERR_STATE, "a symbol or a run length of the BWT does not fit the record widths");
    });
}

// a .rl_bwt image the device accepts: [sb u64][fb u64] in 1..8, then a whole, non-zero number of records
static bool image_ok(const void* image, uint64_t image_bytes) {
    if (image_bytes < 16) return false;
    u64 hdr[2];
    memcpy(hdr, image, 16);
    if (hdr[0] < 1 || hdr[0] > 8 || hdr[1] < 1 || hdr[1] > 8) return false;
    const u64 body = image_bytes - 16;
    return body != 0 && body % (hdr[0] + hdr[1]) == 0;
}

int grlgpu_invert(grlgpu_ctx* ctx, const void* image, uint64_t image_bytes, int cell_bytes, uint64_t n_seqs, void* out, uint64_t cap_bytes, grlgpu_invert_t* info) {
    if (!ctx || !image || !info || !(cell_bytes == 1 || cell_bytes == 2 || cell_bytes == 4 || cell_bytes == 8)) return GRLGPU_ERR_ARG;
    memset(info, 0, sizeof(*info));
    if (!image_ok(image, image_bytes)) return GRLGPU_ERR_ARG;
    if (!out && cap_bytes) return GRLGPU_ERR_ARG;
    return guarded(ctx, [&] { invert_image(ctx, (const u8*)image, image_bytes, cell_bytes, n_seqs, out, cap_bytes, info); });
}

int grlgpu_fm_load(grlgpu_ctx* ctx, const void* image, uint64_t image_bytes, grlgpu_fm_t* info) {
    if (!ctx) return GRLGPU_ERR_ARG;
    ctx->fm.reset();  // the index already loaded goes first: a failed load leaves none
    if (!image || !info) return GRLGPU_ERR_ARG;
    memset(info, 0, sizeof(*info));
    if (!image_ok(image, image_bytes)) return GRLGPU_ERR_ARG;
    return guarded(ctx, [&] { fm_load(ctx, (const u8*)image, image_bytes, info); });
}

// patterns: cell width in {1,2,4,8}, n_pat + 1 offsets from 0, each pattern at least one cell
static int fm_patterns_ok(const void* pat, const uint64_t* pat_off, uint64_t n_pat, int pat_bytes) {
    if (!(pat_bytes == 1 || pat_bytes == 2 || pat_bytes == 4 || pat_bytes == 8)) return GRLGPU_ERR_ARG;
    if (n_pat == 0) return GRLGPU_OK;
    if (!pat || !pat_off || pat_off[0] != 0) return GRLGPU_ERR_ARG;
    for (u64 q = 0; q < n_pat; q++)
        if (pat_off[q + 1] <= pat_off[q]) return GRLGPU_ERR_ARG;
    return GRLGPU_OK;
}

int grlgpu_fm_count(grlgpu_ctx* ctx, const void* pat, const uint64_t* pat_off, uint64_t n_pat, int pat_bytes, uint64_t* sp_ep, grlgpu_fm_query_t* info) {
    if (!ctx || !info) return GRLGPU_ERR_ARG;
    memset(info, 0, sizeof(*info));
    if (const int rc = fm_patterns_ok(pat, pat_off, n_pat, pat_bytes)) return rc;
    if (n_pat && !sp_ep) return GRLGPU_ERR_ARG;
    if (!ctx->fm) return GRLGPU_ERR_STATE;
    if (n_pat == 0) return GRLGPU_OK;
    return guarded(ctx, [&] { fm_query(ctx, pat, pat_off, n_pat, pat_bytes, sp_ep, nullptr, nullptr, nullptr, 0, info); });
}

int grlgpu_fm_locate(grlgpu_ctx* ctx, const void* pat, const uint64_t* pat_off, uint64_t n_pat, int pat_bytes, uint64_t* occ_off, uint32_t* str_id, uint32_t* str_pos,
                     uint64_t cap_occ, grlgpu_fm_query_t* info) {
    if (!ctx || !info) return GRLGPU_ERR_ARG;
    memset(info, 0, sizeof(*info));
    if (const int rc = fm_patterns_ok(pat, pat_off, n_pat, pat_bytes)) return rc;
    if ((n_pat && !occ_off) || (cap_occ && (!str_id || !str_pos))) return GRLGPU_ERR_ARG;
    if (!ctx->fm) return GRLGPU_ERR_STATE;
    if (n_pat == 0) return GRLGPU_OK;
    return guarded(ctx, [&] { fm_query(ctx, pat, pat_off, n_pat, pat_bytes, nullptr, occ_off, str_id, str_pos, cap_occ, info); });
}

int grlgpu_fm_approx_count(grlgpu_ctx* ctx, const void* pat, const uint64_t* pat_off, uint64_t n_pat, int pat_bytes, uint32_t max_mismatches, uint64_t* hit_off,
                           uint64_t* sp_ep, uint8_t* hit_mm, uint64_t cap_hits, grlgpu_fm_approx_t* info) {
    if (!ctx || !info) return GRLGPU_ERR_ARG;
    memset(info, 0, sizeof(*info));
    if (const int rc = fm_patterns_ok(pat, pat_off, n_pat, pat_bytes)) return rc;
    if (max_mismatches > FM_APPROX_MAX_K || (n_pat && !hit_off) || (cap_hits && (!sp_ep || !hit_mm))) return GRLGPU_ERR_ARG;
    if (!ctx->fm) return GRLGPU_ERR_STATE;
    if (n_pat >> 32) return GRLGPU_ERR_LIMIT;
    if (n_pat == 0) return GRLGPU_OK;
    return guarded(ctx, [&] { fm_approx_count(ctx, pat, pat_off, n_pat, pat_bytes, max_mismatches, hit_off, sp_ep, hit_mm, cap_hits, info); });
}

int grlgpu_fm_approx_locate(grlgpu_ctx* ctx, const void* pat, const uint64_t* pat_off, uint64_t n_pat, int pat_bytes, uint32_t max_mismatches, uint64_t* occ_off,
                            uint32_t* str_id, uint32_t* str_pos, uint8_t* occ_mm, uint64_t cap_occ, grlgpu_fm_approx_t* info) {
    if (!ctx || !info) return GRLGPU_ERR_ARG;
    memset(info, 0, sizeof(*info));
    if (const int rc = fm_patterns_ok(pat, pat_off, n_pat, pat_bytes)) return rc;
    if (max_mismatches > FM_APPROX_MAX_K || (n_pat && !occ_off) || (cap_occ && (!str_id || !str_pos || !occ_mm))) return GRLGPU_ERR_ARG;
    if (!ctx->fm) return GRLGPU_ERR_STATE;
    if (n_pat >> 32) return GRLGPU_ERR_LIMIT;
    if (n_pat == 0) return GRLGPU_OK;
    return guarded(ctx, [&] { fm_approx_locate(ctx, pat, pat_off, n_pat, pat_bytes, max_mismatches, occ_off, str_id, str_pos, occ_mm, cap_occ, info); });
}

int grlgpu_fm_extract(grlgpu_ctx* ctx, const uint32_t* str_id, const uint32_t* from, const uint32_t* len, uint64_t n_req, int cell_bytes, uint64_t* out_off, void* out,
                      uint64_t cap_cells, grlgpu_fm_extract_t* info) {
    if (!ctx || !info) return GRLGPU_ERR_ARG;
    memset(info, 0, sizeof(*info));
    if (!(cell_bytes == 1 || cell_bytes == 2 || cell_bytes == 4 || cell_bytes == 8)) return GRLGPU_ERR_ARG;
    if ((n_req && (!str_id || !from || !len || !out_off)) || (cap_cells && !out)) return GRLGPU_ERR_ARG;
    if (!ctx->fm) return GRLGPU_ERR_STATE;
    if (n_req >> 32) return GRLGPU_ERR_LIMIT;
    for (u64 q = 0; q < n_req; q++)
        if (str_id[q] >= ctx->fm->t.N) return GRLGPU_ERR_ARG;
    if (n_req == 0) {
        if (out_off) out_off[0] = 0;
        return GRLGPU_OK;
    }
    return guarded(ctx, [&] { fm_extract(ctx, str_id, from, len, (u32)n_req, cell_bytes, out_off, out, cap_cells, info); });
}

int grlgpu_fm_drop(grlgpu_ctx* ctx) {
    if (!ctx) return GRLGPU_ERR_ARG;
    return guarded(ctx, [&] { ctx->fm.reset(); });
}

int grlgpu_profile_enable(grlgpu_ctx* ctx, int on) {
    if (!ctx) return GRLGPU_ERR_ARG;
    ctx->prof.resolve();
    ctx->prof.timing = on != 0;
    return GRLGPU_OK;
}
int grlgpu_profile_reset(grlgpu_ctx* ctx) {
    if (!ctx) return GRLGPU_ERR_ARG;
    ctx->prof.reset();
    return GRLGPU_OK;
}
uint64_t grlgpu_launch_count(const grlgpu_ctx* ctx) { return ctx ? ctx->prof.launches : 0; }
int grlgpu_profile_entry(grlgpu_ctx* ctx, int index, char* name, int name_cap, uint64_t* launches, double* total_ms, uint64_t* model_bytes) {
    if (!ctx || !name || name_cap <= 0) return GRLGPU_ERR_ARG;
    ctx->prof.resolve();
    if (index < 0 || (size_t)index >= ctx->prof.acc.size()) return 1;
    auto it = ctx->prof.acc.begin();
    std::advance(it, index);
    snprintf(name, (size_t)name_cap, "%s", it->first.c_str());
    if (launches) *launches = it->second.launches;
    if (total_ms) *total_ms = it->second.ms;
    if (model_bytes) *model_bytes = it->second.bytes;
    return GRLGPU_OK;
}

const char* grlgpu_strerror(int status) {
    switch (status) {
        case GRLGPU_OK: return "ok";
        case GRLGPU_ERR_ARG: return "invalid argument";
        case GRLGPU_ERR_ILL_FORMED: return "the collection is ill formed";
        case GRLGPU_ERR_CUDA: return "CUDA error or no usable device";
        case GRLGPU_ERR_NOMEM: return "out of device memory";
        case GRLGPU_ERR_STATE: return "call out of order";
        case GRLGPU_ERR_LIMIT: return "size limit of the device path exceeded";
    }
    return "unknown status";
}
const char* grlgpu_last_error(const grlgpu_ctx* ctx) { return ctx ? ctx->last_error.c_str() : t_last_error.c_str(); }

// ---- self-test hooks ----
int grlgpu_selftest_scan(const uint32_t* in, uint64_t n, uint64_t* out_exclusive, uint64_t* total) {
    return guarded(nullptr, [&] {
        cudaStream_t st = nullptr;
        DevBuf<u32> din(n, st);
        DevBuf<u64> dout(n, st), tot(1, st);
        GRL_CUDA(cudaMemcpy(din.p, in, n * 4, cudaMemcpyHostToDevice));
        exclusive_scan<u32, u64>(din.p, dout.p, n, tot.p, st);
        GRL_CUDA(cudaMemcpy(out_exclusive, dout.p, n * 8, cudaMemcpyDeviceToHost));
        GRL_CUDA(cudaMemcpy(total, tot.p, 8, cudaMemcpyDeviceToHost));
    });
}
int grlgpu_selftest_sort(uint64_t* keys, uint32_t* vals, uint64_t n, int n_bits) {
    return guarded(nullptr, [&] {
        cudaStream_t st = nullptr;
        DevBuf<u64> k(n, st), ka(n, st);
        DevBuf<u32> v(n, st), va(n, st);
        GRL_CUDA(cudaMemcpy(k.p, keys, n * 8, cudaMemcpyHostToDevice));
        GRL_CUDA(cudaMemcpy(v.p, vals, n * 4, cudaMemcpyHostToDevice));
        u64 *kp = k.p, *kap = ka.p;
        u32 *vp = v.p, *vap = va.p;
        radix_sort_pairs(&kp, &vp, &kap, &vap, n, n_bits, st);
        GRL_CUDA(cudaStreamSynchronize(st));
        GRL_CUDA(cudaMemcpy(keys, kp, n * 8, cudaMemcpyDeviceToHost));
        GRL_CUDA(cudaMemcpy(vals, vp, n * 4, cudaMemcpyDeviceToHost));
    });
}
int grlgpu_selftest_compact(const uint32_t* bits, const uint32_t* prev_bits, uint64_t n_bits, uint64_t* out, uint64_t* count) {
    return guarded(nullptr, [&] {
        cudaStream_t st = nullptr;
        const u64 n_words = div_up(n_bits, 32);
        DevBuf<u32> b(n_words, st), pb(n_words, st);
        GRL_CUDA(cudaMemcpy(b.p, bits, n_words * 4, cudaMemcpyHostToDevice));
        if (prev_bits) GRL_CUDA(cudaMemcpy(pb.p, prev_bits, n_words * 4, cudaMemcpyHostToDevice));
        BitmapCompactor bc;
        const u64 cnt = bc.count(b.p, n_bits, st);
        DevBuf<u64> o(cnt, st);
        bc.write<u64>(prev_bits ? pb.p : nullptr, o.p);
        GRL_CUDA(cudaMemcpy(out, o.p, cnt * 8, cudaMemcpyDeviceToHost));
        *count = cnt;
    });
}

}  // extern "C"
