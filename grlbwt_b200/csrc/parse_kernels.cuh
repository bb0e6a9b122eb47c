// Text-side kernels of one parse round (reference: include/parsing_strategies.h:82-145 scan,
// include/exact_algo/exact_par_phase.hpp:14-84 hash / rewrite functors, external/cdt/lib/utils.cpp:100-189 stats).
//
// Text layout in HBM: n cells of CellT (1/2/4/8 bytes, little endian). Round 1: raw symbols
// (rep bit implicitly 1). Later rounds: cell = (rank << 1) | rep. String ends are a bitmap
// (bit i set <=> cell i is the last cell of its string); in round 1 it is derived from cell == sep.
#pragma once
#include "util.cuh"

namespace grl {

// ------------------------------------------------------------------------------------------------
// K0  collection statistics (utils.cpp:100-189): min / max symbol, number of separators, byte histogram
// ------------------------------------------------------------------------------------------------
struct StatsAcc {
    u64 min_sym, max_sym, n_sep;
    u64 hist[256];
};

template <class CellT>
__global__ void __launch_bounds__(256) stats_kernel(const CellT* __restrict__ text, u64 n, CellT sep, StatsAcc* acc) {
    constexpr int VEC = 16 / sizeof(CellT);
    __shared__ u32 sh[256];
    if (sizeof(CellT) == 1) sh[threadIdx.x] = 0;
    __syncthreads();
    u64 mn = ~0ULL, mx = 0, ns = 0;
    const u64 n_vec = n / VEC;
    const uint4* tv = reinterpret_cast<const uint4*>(text);
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += (u64)gridDim.x * blockDim.x) {
        uint4 q = tv[i];
        const CellT* c = reinterpret_cast<const CellT*>(&q);
#pragma unroll
        for (int k = 0; k < VEC; k++) {
            const u64 s = c[k];
            if (sizeof(CellT) == 1) atomicAdd(&sh[s & 255], 1u);
            else { mn = s < mn ? s : mn; mx = s > mx ? s : mx; }
            ns += (c[k] == sep);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < (n - n_vec * VEC)) {  // tail cells
        const u64 s = text[n_vec * VEC + threadIdx.x];
        if (sizeof(CellT) == 1) atomicAdd(&sh[s & 255], 1u);
        else { mn = s < mn ? s : mn; mx = s > mx ? s : mx; }
        ns += (s == (u64)sep);
    }
    ns = warp_sum(ns);
    if (lane_id() == 0 && ns) atomicAdd(&acc->n_sep, ns);
    if (sizeof(CellT) == 1) {
        __syncthreads();
        if (sh[threadIdx.x]) atomicAdd(&acc->hist[threadIdx.x], (u64)sh[threadIdx.x]);
    } else {
        mn = warp_min(mn);
        mx = warp_max(mx);
        if (lane_id() == 0) { atomicMin(&acc->min_sym, mn); atomicMax(&acc->max_sym, mx); }
    }
}

// ------------------------------------------------------------------------------------------------
// K1  LMS phrase-start flags (parsing_strategies.h:112-138; data-parallel form of SURVEY.md App. H).
// One thread = 32 consecutive cells = one word of the output bitmaps. type[i] (S=1 / L=0) is
// resolved inside the thread where possible, else by the first determined cell to the right:
// ballot inside the warp, shared memory across warps, bounded look-ahead past the CTA; a run of
// equal cells longer than the look-ahead raises *need_slow and the host re-runs with per-CTA
// incoming types computed by the summary/resolve kernels (MODE 1 / lms_resolve_kernel / MODE 2).
// ------------------------------------------------------------------------------------------------
constexpr int LMS_THREADS = 256;
constexpr int LMS_CELLS = 32;
constexpr int LMS_LOOKAHEAD = 128;
enum { ST_L = 0, ST_S = 1, ST_PASS = 2 };

template <class CellT, bool FIRST>
__device__ __forceinline__ u64 cell_value(CellT c) { return FIRST ? (u64)c : ((u64)c >> 1); }

template <class CellT, bool FIRST>
__device__ __forceinline__ bool cell_is_end(const CellT* __restrict__ text, const u32* __restrict__ end_bits, CellT sep, u64 i) {
    if (FIRST) return text[i] == sep;
    return (end_bits[i >> 5] >> (i & 31)) & 1u;
}

// MODE 0: flags with bounded look-ahead; MODE 1: only the per-CTA summary state; MODE 2: flags with given incoming types
template <class CellT, bool FIRST, int MODE>
__global__ void __launch_bounds__(LMS_THREADS) lms_flags_kernel(const CellT* __restrict__ text, u64 n, CellT sep, const u32* __restrict__ end_bits_in,
                                                                u32* __restrict__ end_bits_out, u32* __restrict__ start_bits,
                                                                u8* __restrict__ block_state, const u8* __restrict__ block_incoming, u32* need_slow) {
    __shared__ u32 s_warp[LMS_THREADS / 32];
    __shared__ u32 s_xblk;
    const u64 word = (u64)blockIdx.x * LMS_THREADS + threadIdx.x;
    const u64 base = word * LMS_CELLS;
    const u32 lane = lane_id(), warp = threadIdx.x >> 5;

    // ---- CTA incoming type: type of the first cell after this CTA's range ----
    if (threadIdx.x == LMS_THREADS - 1) {
        u32 x = ST_L;
        if (MODE == 2) x = block_incoming[blockIdx.x];
        else if (MODE == 0) {
            u64 q = ((u64)blockIdx.x + 1) * LMS_THREADS * LMS_CELLS;
            if (q < n) {
                x = ST_PASS;
                for (int k = 0; k < LMS_LOOKAHEAD; k++, q++) {
                    if (cell_is_end<CellT, FIRST>(text, end_bits_in, sep, q)) { x = ST_L; break; }
                    const u64 a = cell_value<CellT, FIRST>(text[q]), b = cell_value<CellT, FIRST>(text[q + 1]);
                    if (a != b) { x = a < b ? ST_S : ST_L; break; }
                }
                if (x == ST_PASS) { atomicExch(need_slow, 1u); x = ST_L; }
            }
        }
        s_xblk = x;
    }

    // ---- load 32 cells; per-cell determined/value masks ----
    u32 valid = 0, endm = 0, repm = 0, detm = 0, valm = 0, gtprev = 0;
    u32 left_end = 1, left_rep = 1;  // position 0 starts a string
    if (base < n) {
        const u64 cnt = n - base;
        valid = cnt >= 32 ? 0xffffffffu : ((1u << cnt) - 1u);
        __align__(16) CellT c[LMS_CELLS];
        if (cnt >= 32) {
            constexpr int NV = LMS_CELLS * sizeof(CellT) / 16;
            const uint4* src = reinterpret_cast<const uint4*>(text + base);
            uint4* dst = reinterpret_cast<uint4*>(c);
#pragma unroll
            for (int k = 0; k < NV; k++) dst[k] = src[k];
        } else {
#pragma unroll
            for (int k = 0; k < LMS_CELLS; k++) c[k] = (u64)k < cnt ? text[base + k] : sep;
        }
        if (FIRST) {
            if constexpr (sizeof(CellT) == 1) {
                u32 w[8];
                memcpy(w, c, 32);
                const u32 sep4 = (u32)sep * 0x01010101u;
#pragma unroll
                for (int j = 0; j < 8; j++) endm |= (((__vcmpeq4(w[j], sep4) & 0x80808080u) * 0x00204081u) >> 28) << (4 * j);
            } else {
#pragma unroll
                for (int k = 0; k < LMS_CELLS; k++) endm |= (u32)(c[k] == sep) << k;
            }
            repm = 0xffffffffu;
        } else {
            endm = end_bits_in[word];
#pragma unroll
            for (int k = 0; k < LMS_CELLS; k++) repm |= (u32)(c[k] & 1) << k;
        }
        endm = (endm & valid) | ~valid;  // cells past the end behave as string ends
        u64 vnext = 0;
        if (cnt > 32) vnext = cell_value<CellT, FIRST>(text[base + 32]);
        u64 vleft = 0;
        if (base > 0) {
            const CellT cl = text[base - 1];
            vleft = cell_value<CellT, FIRST>(cl);
            left_rep = FIRST ? 1u : (u32)(cl & 1);
            left_end = FIRST ? (u32)(cl == sep) : (end_bits_in[word - 1] >> 31);
        }
        if constexpr (sizeof(CellT) == 1 && FIRST) {
            // byte alphabets, round 1 (the 7.5 GB pass of C2): four cells per 32-bit word, byte-wise SIMD compares, and the top bit of
            // every byte gathered into a 4-bit mask by one multiply -- a third of the instructions of the cell-by-cell loop below
            u32 w[8];
            memcpy(w, c, 32);
            const u32 sep4 = (u32)sep * 0x01010101u;
            detm = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const u32 nx = (w[j] >> 8) | ((j < 7 ? w[j + 1] : (u32)vnext) << 24);
                const u32 pv = (w[j] << 8) | (j > 0 ? (w[j - 1] >> 24) : (u32)vleft);
                const u32 e4 = __vcmpeq4(w[j], sep4);
                const u32 d4 = e4 | __vcmpne4(w[j], nx);
                const u32 v4 = __vcmpltu4(w[j], nx) & ~e4;
                const u32 g4 = __vcmpgtu4(pv, w[j]);
                detm |= (((d4 & 0x80808080u) * 0x00204081u) >> 28) << (4 * j);
                valm |= (((v4 & 0x80808080u) * 0x00204081u) >> 28) << (4 * j);
                gtprev |= (((g4 & 0x80808080u) * 0x00204081u) >> 28) << (4 * j);
            }
            // (cells past the end of the text were loaded as separators, so endm -- forced above for them -- already agrees with e4)
            detm |= endm;
            valm &= ~endm;
        } else {
#pragma unroll
        for (int k = 0; k < LMS_CELLS; k++) {
            const u64 v = cell_value<CellT, FIRST>(c[k]);
            const u64 nv = k == LMS_CELLS - 1 ? vnext : cell_value<CellT, FIRST>(c[k == LMS_CELLS - 1 ? k : k + 1]);
            const u64 pv = k == 0 ? vleft : cell_value<CellT, FIRST>(c[k == 0 ? 0 : k - 1]);
            const bool e = (endm >> k) & 1u;
            detm |= (u32)(e || v != nv) << k;
            valm |= (u32)(!e && v < nv) << k;
            gtprev |= (u32)(pv > v) << k;
        }
        }
    } else {
        detm = 0xffffffffu;  // out of range: determined, L
        endm = 0xffffffffu;
    }

    // ---- thread summary and incoming type ----
    const u32 my_state = detm ? ((valm >> (__ffs(detm) - 1)) & 1u) : (u32)ST_PASS;
    const u32 nonpass = __ballot_sync(0xffffffffu, my_state != ST_PASS);
    const u32 sbits = __ballot_sync(0xffffffffu, my_state == ST_S);
    if (lane == 0) s_warp[warp] = nonpass ? ((sbits >> (__ffs(nonpass) - 1)) & 1u) : (u32)ST_PASS;
    __syncthreads();
    if (MODE == 1) {
        if (threadIdx.x == 0) {
            u32 st = ST_PASS;
            for (int w = 0; w < LMS_THREADS / 32; w++)
                if (s_warp[w] != ST_PASS) { st = s_warp[w]; break; }
            block_state[blockIdx.x] = (u8)st;
        }
        return;
    }
    u32 x;
    {
        const u32 m = lane == 31 ? 0u : (nonpass & ~((2u << lane) - 1u));
        if (m) x = (sbits >> (__ffs(m) - 1)) & 1u;
        else {
            x = ST_PASS;
            for (int w = warp + 1; w < LMS_THREADS / 32; w++)
                if (s_warp[w] != ST_PASS) { x = s_warp[w]; break; }
            if (x == ST_PASS) x = s_xblk;
        }
    }
    if (base >= n) return;

    // ---- types of own cells: type(k) = det(k) ? val(k) : type(k+1), type(32) = x ----
    u32 typem = 0, t = x;
#pragma unroll
    for (int k = LMS_CELLS - 1; k >= 0; k--) {
        t = ((detm >> k) & 1u) ? ((valm >> k) & 1u) : t;
        typem |= t << k;
    }
    const u32 real_end = endm & valid;
    const u32 prev_end = (real_end << 1) | left_end;   // is_start(k): k begins a string
    const u32 prev_rep = (repm << 1) | left_rep;
    const u32 brk = gtprev & typem & repm & prev_rep & ~prev_end;  // parsing_strategies.h:121-123
    start_bits[word] = (prev_end | brk) & valid;
    if (FIRST) end_bits_out[word] = real_end;
}

// serial reverse pass over the per-CTA summary states (slow path only; one thread)
static __global__ void lms_resolve_kernel(const u8* __restrict__ block_state, u8* __restrict__ block_incoming, u64 n_blocks) {
    if (blockIdx.x || threadIdx.x) return;
    u8 inc = ST_L;
    for (u64 b = n_blocks; b-- > 0;) {
        block_incoming[b] = inc;
        if (block_state[b] != ST_PASS) inc = block_state[b];
    }
}

// ------------------------------------------------------------------------------------------------
// K3  phrase deduplication + counting (ext_hash_functor exact_par_phase.hpp:33-39; replaces the
// XXH3-keyed Robin-Hood table hash_table.hpp:451-539).
//
// Global table: open addressing, linear probing, 16-byte entries {key = first-occurrence position << 24 |
// min(len, LEN_SAT), count}; a key is claimed with one 64-bit CAS and is immediately complete because it
// points into the immutable text.
//
// dedup_cached_kernel is the fused text pass: persistent CTAs walk 32 KB tiles of cells staged in shared memory
// (cells + look-ahead halo, start/end bitmap words); a thread owns one bitmap word, numbers its phrases
// from the tile's scanned base and, for phrases of at most 15 bytes, packs the cells into a 128-bit key
// and looks it up in a per-CTA shared-memory cache of hot phrases (key -> global slot, local count).
// Hits cost shared memory only; counts are flushed to the global table once per CTA. Misses and longer
// phrases take the global path (hash of the cells, probe, compare against the first occurrence).
// ------------------------------------------------------------------------------------------------
constexpr u64 HT_EMPTY = ~0ULL;
constexpr u64 HT_LEN_SAT = 0xFFFFFFULL;
constexpr int HT_MAX_PROBES = 512;
constexpr u32 HT_OVERFLOW = 0xffffffffu;

// smallest position q > pos that starts a phrase, or n (the virtual start after the last cell)
__device__ __forceinline__ u64 next_start_after(const u32* __restrict__ start_bits, u64 n, u64 pos) {
    const u64 n_words = (n + 31) >> 5;
    u64 q = pos + 1;
    if (q >= n) return n;
    u64 w = q >> 5;
    u32 x = start_bits[w] & (0xffffffffu << (q & 31));
    while (!x) {
        if (++w >= n_words) return n;
        x = start_bits[w];
    }
    q = (w << 5) + (u64)(__ffs(x) - 1);
    return q < n ? q : n;
}
__device__ __forceinline__ bool bit_at(const u32* __restrict__ bits, u64 i) { return (bits[i >> 5] >> (i & 31)) & 1u; }

// true length of the phrase that starts at pos (closed interval; the last phrase of a string stops at the string end)
__device__ __forceinline__ u64 phrase_len_bits(const u32* __restrict__ start_bits, const u32* __restrict__ end_bits, u64 n, u64 pos) {
    const u64 q = next_start_after(start_bits, n, pos);
    return bit_at(end_bits, q - 1) ? q - pos : q - pos + 1;
}

template <class CellT>
__device__ __forceinline__ u64 phrase_hash(const CellT* __restrict__ text, u64 s, u64 len) {
    u64 h = 0xcbf29ce484222325ULL ^ len;
    for (u64 i = 0; i < len; i++) h = (h ^ (u64)text[s + i]) * 0x100000001b3ULL;
    return mix64(h);
}

// global path: probes `table` (whose keys point into ttext) for the phrase qtext[s, s+len), claims a slot if the
// phrase is new (then qtext must be ttext) and adds `add` to its count; returns the slot, or HT_OVERFLOW when the
// probe limit is hit.
template <class CellT>
__device__ u32 table_probe(const CellT* __restrict__ qtext, u64 s, u64 len, const CellT* __restrict__ ttext, ulonglong2* table, u64 cap, u64 add,
                           const u32* __restrict__ start_bits, const u32* __restrict__ end_bits, u64 n, u32* overflow) {
    const u64 lenf = len < HT_LEN_SAT ? len : HT_LEN_SAT;
    const u64 mykey = (s << 24) | lenf;
    u64 slot = __umul64hi(phrase_hash<CellT>(qtext, s, len), cap);  // uniform over [0, cap), cap need not be a power of two
    for (int probes = 0; probes < HT_MAX_PROBES; probes++) {
        u64 k = *reinterpret_cast<volatile u64*>(&table[slot].x);
        if (k == HT_EMPTY) {
            const u64 old = atomicCAS(&table[slot].x, HT_EMPTY, mykey);
            k = old == HT_EMPTY ? mykey : old;
        }
        bool match = k == mykey;
        if (!match && (k & HT_LEN_SAT) == lenf) {
            const u64 kpos = k >> 24;
            match = true;
            for (u64 i = 0; i < len; i++)
                if (ttext[kpos + i] != qtext[s + i]) { match = false; break; }
            if (match && lenf == HT_LEN_SAT) match = start_bits != nullptr && phrase_len_bits(start_bits, end_bits, n, kpos) == len;
        }
        if (match) {
            atomicAdd(&table[slot].y, add);
            return (u32)slot;
        }
        if (++slot == cap) slot = 0;
    }
    atomicExch(overflow, 1u);
    return HT_OVERFLOW;
}
template <class CellT>
__device__ __forceinline__ u32 table_insert_global(const CellT* __restrict__ text, u64 s, u64 len, ulonglong2* table, u64 cap, const u32* __restrict__ start_bits,
                                                   const u32* __restrict__ end_bits, u64 n, u32* overflow) {
    return table_probe<CellT>(text, s, len, text, table, cap, 1ULL, start_bits, end_bits, n, overflow);
}

// ---- thread-per-phrase variant over a compacted start array (unique-heavy rounds: maximum memory-level parallelism) ----
template <class PosT>
struct PosFlag {
    static constexpr PosT FLAG = PosT(1) << (sizeof(PosT) * 8 - 1);
};
// phrase j covers [s, e] (closed); fin = it is the last phrase of its string (parsing_strategies.h:126,141)
template <class PosT>
__device__ __forceinline__ void phrase_span(const PosT* __restrict__ ps, u64 j, u64& s, u64& e, bool& fin) {
    constexpr PosT FLAG = PosFlag<PosT>::FLAG;
    const PosT a = ps[j], b = ps[j + 1];
    s = (u64)(a & ~FLAG);
    fin = (b & FLAG) != 0;
    e = fin ? (u64)(b & ~FLAG) - 1 : (u64)(b & ~FLAG);
}
template <class CellT, class PosT>
__global__ void __launch_bounds__(256) phrase_insert_kernel(const CellT* __restrict__ text, u64 n, const PosT* __restrict__ ps, u64 j0, u64 p,
                                                            const u32* __restrict__ start_bits, const u32* __restrict__ end_bits, ulonglong2* table,
                                                            u64 cap, u32* __restrict__ slot_of_phrase, u32* overflow) {
    const u64 j = j0 + (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= p) return;
    if (*reinterpret_cast<volatile u32*>(overflow)) return;  // the table is too small: the host regrows it and redoes the pass
    u64 s, e; bool fin;
    phrase_span<PosT>(ps, j, s, e, fin);
    const u32 slot = table_insert_global<CellT>(text, s, e - s + 1, table, cap, start_bits, end_bits, n, overflow);
    slot_of_phrase[j] = (slot & 0x7fffffffu) | (fin ? 0x80000000u : 0u);
}

// ---- fused, cached variant (duplicate-heavy rounds) ----
constexpr int FD_THREADS = 1024;               // one CTA per SM (2 x 512 threads with half-size tiles and caches measured the same)
constexpr int FD_CTAS_PER_SM = 1;
constexpr int FD_TILE_BYTES = 32768;           // staged cells per tile: 32768 / sizeof(CellT) cells
constexpr int FD_HALO_WORDS = 4;               // look-ahead for the end of a tile's last phrases: 128 cells
constexpr int FD_HALO = FD_HALO_WORDS * 32;
constexpr int FD_LIST_CAP = 16384;             // phrase starts of one tile (u16 tile-local positions)
constexpr int FD_MISS_CAP = 8192;              // deferred phrases of one tile
constexpr int FD_CACHE = 4096;                 // hot-phrase cache entries per CTA, 2-way
constexpr int FD_CACHE_BITS = 12;
constexpr u32 FD_NONE = 0xffffffffu;

template <class CellT>
__host__ __device__ constexpr int fd_tile_words() { return FD_TILE_BYTES / 32 / (int)sizeof(CellT); }  // bitmap words per tile
template <class CellT>
__host__ __device__ constexpr size_t fd_cell_bytes() { return (size_t)FD_TILE_BYTES + (size_t)FD_HALO * sizeof(CellT) + 32; }  // + slack for the 3 x u64 window
template <class CellT>
__host__ __device__ constexpr size_t fd_smem_bytes() {
    return fd_cell_bytes<CellT>() + 2 * (size_t)(fd_tile_words<CellT>() + FD_HALO_WORDS) * sizeof(u32)  // cells, start / end words
           + (size_t)FD_LIST_CAP * 2 + (size_t)FD_MISS_CAP * 2                                         // start list, deferred list
           + (size_t)FD_CACHE * (8 + 8 + 4 + 4 + 4)                                                     // cache: k0, k1, slot, count, state
           + 64 * sizeof(u32);                                                                          // scan scratch + scalars
}

// per-tile phrase counts (tile = words_per_tile bitmap words)
static __global__ void __launch_bounds__(256) tile_popc_kernel(const u32* __restrict__ start_bits, u64 n_words, int words_per_tile, u32* __restrict__ tile_cnt) {
    __shared__ u32 sm[33];
    const u64 w0 = (u64)blockIdx.x * words_per_tile;
    u32 c = 0, tot;
    for (int k = threadIdx.x; k < words_per_tile; k += 256)
        if (w0 + k < n_words) c += __popc(start_bits[w0 + k]);
    block_exclusive_sum<u32>(c, sm, tot);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = tot;
}

// 128-bit key of the phrase cells[sl, sl+len): its bytes, little endian, length in the top byte (len * W <= 15)
template <int W>
__device__ __forceinline__ void fd_pack_key(const unsigned char* s_cells, u32 sl, u64 len, u64& k0, u64& k1) {
    const u32 bo = sl * W, sh = (bo & 7u) * 8u;
    const u64 nb = len * W;
    const u64* q8 = reinterpret_cast<const u64*>(s_cells + (bo & ~7u));
    const u64 w0 = q8[0], w1 = q8[1], w2 = q8[2];
    k0 = sh ? ((w0 >> sh) | (w1 << (64 - sh))) : w0;
    k1 = sh ? ((w1 >> sh) | (w2 << (64 - sh))) : w1;
    if (nb < 8) { k0 &= (1ULL << (nb * 8)) - 1ULL; k1 = 0; }
    else if (nb == 8) k1 = 0;
    else k1 &= (1ULL << ((nb - 8) * 8)) - 1ULL;
    k1 |= len << 56;
}

// stats[0] += phrases that took the global path, stats[1] += phrases seen (the host reads them after a pilot launch)
template <class CellT>
__global__ void __launch_bounds__(FD_THREADS, FD_CTAS_PER_SM) dedup_cached_kernel(const CellT* __restrict__ text, u64 n, const u32* __restrict__ start_bits,
                                                                     const u32* __restrict__ end_bits, const u64* __restrict__ tile_base, u64 t_begin,
                                                                     u64 t_end, ulonglong2* table, u64 cap, u32* __restrict__ slot_of_phrase,
                                                                     u32* overflow, u64* stats) {
    extern __shared__ __align__(16) unsigned char fd_smem[];
    constexpr int W = sizeof(CellT);
    constexpr int TW = fd_tile_words<CellT>();
    constexpr int NW = TW + FD_HALO_WORDS;
    constexpr int TILE = TW * 32;
    unsigned char* s_cells = fd_smem;
    u32* s_start = reinterpret_cast<u32*>(fd_smem + fd_cell_bytes<CellT>());
    u32* s_end = s_start + NW;
    u16* s_list = reinterpret_cast<u16*>(s_end + NW);
    u16* s_miss = s_list + FD_LIST_CAP;
    volatile u64* c_k0 = reinterpret_cast<volatile u64*>(s_miss + FD_MISS_CAP);
    volatile u64* c_k1 = c_k0 + FD_CACHE;
    volatile u32* c_slot = reinterpret_cast<volatile u32*>(c_k1 + FD_CACHE);
    volatile u32* c_cnt = c_slot + FD_CACHE;
    volatile u32* c_state = c_cnt + FD_CACHE;
    u32* s_scan = const_cast<u32*>(c_state) + FD_CACHE;  // [0..32] scan scratch, [40] abort, [41] tail next, [42] deferred count
    const u64 n_words = (n + 31) >> 5;
    u64 my_global = 0, my_seen = 0;
    for (int i = threadIdx.x; i < FD_CACHE; i += FD_THREADS) { c_state[i] = 0; c_cnt[i] = 0; }
    // "table too small" flag: thread 0 reads it one tile ahead, so the load's latency hides behind a tile's work instead of stalling
    // all 1024 threads at the barrier below (27 % of the kernel's stall samples in the round-2 ncu capture)
    u32 ovf_ahead = 0;
    if (threadIdx.x == 0) ovf_ahead = *reinterpret_cast<volatile u32*>(overflow);

    for (u64 t = t_begin + blockIdx.x; t < t_end; t += gridDim.x) {
        if (threadIdx.x == 0) {
            s_scan[40] = ovf_ahead;
            s_scan[42] = 0;
            ovf_ahead = *reinterpret_cast<volatile u32*>(overflow);
        }
        __syncthreads();  // also orders the previous tile's shared-memory reads before this tile's loads
        if (s_scan[40]) break;  // the table is too small: the host regrows it and redoes the pass
        const u64 tile0 = t * TILE, word0 = t * TW;
        // ---- P0: stage cells (16-byte vectors) and bitmap words ----
        {
            const u64 cells_here = (n - tile0) < (u64)(TILE + FD_HALO) ? (n - tile0) : (u64)(TILE + FD_HALO);
            const u64 bytes = cells_here * W, nvec = bytes >> 4;
            const unsigned char* tsrc = reinterpret_cast<const unsigned char*>(text) + tile0 * W;
            const uint4* src = reinterpret_cast<const uint4*>(tsrc);
            uint4* dst = reinterpret_cast<uint4*>(s_cells);
            for (u64 v = threadIdx.x; v < nvec; v += FD_THREADS) dst[v] = src[v];
            for (u64 b = (nvec << 4) + threadIdx.x; b < bytes; b += FD_THREADS) s_cells[b] = tsrc[b];
        }
        for (int k = threadIdx.x; k < NW; k += FD_THREADS) {
            const u64 wi = word0 + k;
            s_start[k] = wi < n_words ? start_bits[wi] : 0u;
            s_end[k] = wi < n_words ? end_bits[wi] : 0u;
        }
        __syncthreads();
        // ---- P1: tile-local positions of the phrase starts, in order ----
        const u32 mine = (int)threadIdx.x < TW ? s_start[threadIdx.x] : 0u;  // real starts (bits >= n are zero in the bitmap)
        u32 tot;
        const u32 pre = block_exclusive_sum<u32>(__popc(mine), s_scan, tot);
        if (threadIdx.x == 0) {
            const u64 vw = n >> 5;  // position n acts as a start so the last phrase finds its end
            if (vw >= word0 && vw < word0 + NW) s_start[vw - word0] |= 1u << (n & 31);
            u32 tn = FD_NONE;
            for (int k = TW; k < NW; k++)
                if (s_start[k]) { tn = k * 32 + (__ffs(s_start[k]) - 1); break; }
            s_scan[41] = tn;
        }
        const u64 jbase = tile_base[t];
        if (tot <= (u32)FD_LIST_CAP) {
            u32 x = mine, o = pre;
            while (x) { s_list[o++] = (u16)(threadIdx.x * 32 + (__ffs(x) - 1)); x &= x - 1; }
        }
        __syncthreads();
        my_seen += (threadIdx.x == 0) ? tot : 0;
        if (tot > (u32)FD_LIST_CAP) {
            // pathological tile (more starts than the list holds, e.g. runs of empty strings): owner-thread loop, global path
            u32 x = mine;
            u64 j = jbase + pre;
            while (x) {
                const u32 b = __ffs(x) - 1;
                x &= x - 1;
                const u64 s = tile0 + threadIdx.x * 32 + b;
                const u64 q = next_start_after(start_bits, n, s);
                const bool fin = bit_at(end_bits, q - 1);
                const u32 slot = table_insert_global<CellT>(text, s, (fin ? q - 1 : q) - s + 1, table, cap, start_bits, end_bits, n, overflow);
                slot_of_phrase[j++] = (slot & 0x7fffffffu) | (fin ? 0x80000000u : 0u);
                my_global++;
            }
            continue;
        }
        const u32 tail_next = s_scan[41];
        // ---- P2a: one phrase per thread and step; cache hits finish here, everything else is deferred ----
        for (u32 k = threadIdx.x; k < tot; k += FD_THREADS) {
            const u32 sl = s_list[k];
            const u32 nl = k + 1 < tot ? (u32)s_list[k + 1] : tail_next;
            bool done = false;
            if (nl != FD_NONE) {
                const bool fin = (s_end[(nl - 1) >> 5] >> ((nl - 1) & 31)) & 1u;
                const u64 len = (u64)(fin ? nl - 1 : nl) - sl + 1;
                if (len * W <= 15) {
                    u64 k0, k1;
                    fd_pack_key<W>(s_cells, sl, len, k0, k1);
                    const u32 ci = (u32)(((k0 ^ (k1 * 0x9E3779B97F4A7C15ULL)) * 0xff51afd7ed558ccdULL) >> (64 - FD_CACHE_BITS));
#pragma unroll
                    for (int way = 0; way < 2; way++) {
                        const u32 c = ci ^ (u32)way;
                        if (!done && c_state[c] == 2u && c_k0[c] == k0 && c_k1[c] == k1) {
                            atomicAdd(const_cast<u32*>(&c_cnt[c]), 1u);
                            slot_of_phrase[jbase + k] = (c_slot[c] & 0x7fffffffu) | (fin ? 0x80000000u : 0u);
                            done = true;
                        }
                    }
                }
            }
            if (!done) {
                const u32 m = atomicAdd(&s_scan[42], 1u);
                if (m < (u32)FD_MISS_CAP) s_miss[m] = (u16)k;
                else {  // deferred list full: take the global path right away
                    u64 s = tile0 + sl, q = nl != FD_NONE ? tile0 + nl : next_start_after(start_bits, n, s);
                    const bool fin = bit_at(end_bits, q - 1);
                    const u32 slot = table_insert_global<CellT>(text, s, (fin ? q - 1 : q) - s + 1, table, cap, start_bits, end_bits, n, overflow);
                    slot_of_phrase[jbase + k] = (slot & 0x7fffffffu) | (fin ? 0x80000000u : 0u);
                    my_global++;
                }
            }
        }
        __syncthreads();
        // ---- P2b: deferred phrases: global table, then try to cache the key ----
        const u32 n_def = s_scan[42] < (u32)FD_MISS_CAP ? s_scan[42] : (u32)FD_MISS_CAP;
        for (u32 m = threadIdx.x; m < n_def; m += FD_THREADS) {
            const u32 k = s_miss[m];
            const u32 sl = s_list[k];
            const u32 nl = k + 1 < tot ? (u32)s_list[k + 1] : tail_next;
            const u64 s = tile0 + sl, q = nl != FD_NONE ? tile0 + nl : next_start_after(start_bits, n, s);
            const bool fin = bit_at(end_bits, q - 1);
            const u64 len = (fin ? q - 1 : q) - s + 1;
            const u32 slot = table_insert_global<CellT>(text, s, len, table, cap, start_bits, end_bits, n, overflow);
            slot_of_phrase[jbase + k] = (slot & 0x7fffffffu) | (fin ? 0x80000000u : 0u);
            my_global++;
            if (nl != FD_NONE && len * W <= 15 && slot != HT_OVERFLOW) {
                u64 k0, k1;
                fd_pack_key<W>(s_cells, sl, len, k0, k1);
                const u32 ci = (u32)(((k0 ^ (k1 * 0x9E3779B97F4A7C15ULL)) * 0xff51afd7ed558ccdULL) >> (64 - FD_CACHE_BITS));
                for (int way = 0; way < 2; way++) {
                    const u32 c = ci ^ (u32)way;
                    // the cache words are the only locations two threads of this phase touch without a barrier in between (this is the
                    // miss path): every access to them is an atomic -- the state word acquires (a read-modify-write that changes
                    // nothing) and releases (fence, then exchange) the key and slot words written by the thread that claimed the way
                    const u32 stt = atomicOr(const_cast<u32*>(&c_state[c]), 0u);
                    if (stt == 2u && atomicOr(const_cast<u64*>(&c_k0[c]), 0ULL) == k0 && atomicOr(const_cast<u64*>(&c_k1[c]), 0ULL) == k1) break;  // cached meanwhile
                    if (stt == 0u && atomicCAS(const_cast<u32*>(&c_state[c]), 0u, 1u) == 0u) {
                        atomicExch(const_cast<u64*>(&c_k0[c]), k0);
                        atomicExch(const_cast<u64*>(&c_k1[c]), k1);
                        atomicExch(const_cast<u32*>(&c_slot[c]), slot);
                        __threadfence_block();
                        atomicExch(const_cast<u32*>(&c_state[c]), 2u);
                        break;
                    }
                }
            }
        }
    }
    // ---- flush the cached counts and the pilot statistics ----
    __syncthreads();
    for (int i = threadIdx.x; i < FD_CACHE; i += FD_THREADS)
        if (c_state[i] == 2u && c_cnt[i]) atomicAdd(&table[c_slot[i]].y, (u64)c_cnt[i]);
    if (stats) {
        if (my_global) atomicAdd(&stats[0], my_global);
        if (my_seen) atomicAdd(&stats[1], my_seen);
    }
}

static __global__ void __launch_bounds__(256) table_occupancy_kernel(const ulonglong2* __restrict__ table, u64 cap, u32* __restrict__ occ_bits) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;  // cap is a multiple of 256
    const u32 b = __ballot_sync(0xffffffffu, table[i].x != HT_EMPTY);
    if (lane_id() == 0) occ_bits[i >> 5] = b;
}

// ------------------------------------------------------------------------------------------------
// Multi-GPU exchange helpers (SURVEY.md 8e): a "pack" is a list of phrases as (lens[m], counts[m], cells
// concatenated); packs travel between ranks, and the same table code dedups them by treating the pack's
// cell buffer as the text the keys point into.
// ------------------------------------------------------------------------------------------------
template <class CellT>
__global__ void __launch_bounds__(256) phrase_owner_kernel(const CellT* __restrict__ text, const u64* __restrict__ ph_pos, const u32* __restrict__ ph_len, u64 d,
                                                           u32 n_ranks, u64* __restrict__ keys, u32* __restrict__ vals) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d) return;
    keys[i] = phrase_hash<CellT>(text, ph_pos[i], ph_len[i]) % n_ranks;  // content hash: the same owner on every rank
    vals[i] = (u32)i;
}
static __global__ void gather_u32_kernel(const u32* __restrict__ src, const u32* __restrict__ perm, u64 m, u32* __restrict__ dst) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < m) dst[k] = src[perm[k]];
}
// dedup of a pack into a table whose keys point into the pack's own cells; count += counts[k] (or the index k when counts == nullptr)
template <class CellT>
__global__ void __launch_bounds__(256) pack_insert_kernel(const CellT* __restrict__ cells, const u64* __restrict__ offs, const u32* __restrict__ lens,
                                                          const u64* __restrict__ counts, u64 m, ulonglong2* table, u64 cap, u32* overflow,
                                                          u32* __restrict__ slot_out) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    if (*reinterpret_cast<volatile u32*>(overflow)) return;
    const u32 slot = table_probe<CellT>(cells, offs[k], lens[k], cells, table, cap, counts ? counts[k] : k, nullptr, nullptr, 0, overflow);
    if (slot_out) slot_out[k] = slot;
}
// owner side of the metasymbol return: dense partition index of every table slot, then of every received phrase
static __global__ void __launch_bounds__(256) slot_dense_kernel(const u32* __restrict__ pslots, u64 d_part, ulonglong2* table) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < d_part) table[pslots[i]].y = i;
}
static __global__ void __launch_bounds__(256) recv_dense_kernel(const u32* __restrict__ recv_slot, u64 m, const ulonglong2* __restrict__ table, u32* __restrict__ dense) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < m) dense[k] = (u32)table[recv_slot[k]].y;
}
static __global__ void __launch_bounds__(256) reply_meta_kernel(const u32* __restrict__ dense, u64 m, u64 part_base, const u64* __restrict__ g_meta, u64* __restrict__ reply) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < m) reply[k] = g_meta[part_base + dense[k]];
}
// requester side: the k-th returned metasymbol belongs to the k-th phrase of the pack this rank sent (owner order)
static __global__ void __launch_bounds__(256) apply_reply_kernel(const u32* __restrict__ perm, const u32* __restrict__ occ_slots, const u64* __restrict__ local_meta, u64 d,
                                                                 ulonglong2* ltable) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < d) ltable[occ_slots[perm[k]]].y = local_meta[k];
}

// ------------------------------------------------------------------------------------------------
// K7  rewrite (ext_parse_functor exact_par_phase.hpp:53-59, parse_text parsing_strategies.h:644-676):
// out[j] = metasymbol of phrase occurrence j (stored in the entry's count field by then), forward
// order; the string-end bitmap of the new text comes from the per-occurrence "final" flag.
// ------------------------------------------------------------------------------------------------
template <class OutT>
__global__ void __launch_bounds__(256) rewrite_kernel(const u32* __restrict__ slot_of_phrase, u64 p, const ulonglong2* __restrict__ table,
                                                      OutT* __restrict__ out, u32* __restrict__ end_bits_out) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u32 fin = 0;
    if (j < p) {
        const u32 sv = slot_of_phrase[j];
        fin = sv >> 31;
        out[j] = (OutT)ld_gather8(&table[sv & 0x7fffffffu].y);
    }
    const u32 b = __ballot_sync(0xffffffffu, fin);
    if (lane_id() == 0 && (j >> 5) < ((p + 31) >> 5)) end_bits_out[j >> 5] = b;
}

}  // namespace grl
