// Dictionary-side kernels of one parse round: compaction of the phrase table into a contiguous
// dictionary (exact_par_phase.hpp:106-183), ordering of ALL dictionary suffixes under the
// "proper prefix is greater" order with equal-suffix grouping (what suffix_induction,
// exact_LMS_induction.h:94-158, produces), ranks among unsolved blocks + preliminary BWT
// (produce_pre_bwt, exact_par_phase.cpp:136-242), grammar rules (produce_grammar, :14-95) and
// metasymbol assignment (:427-450).
//
// Dictionary layout in HBM (structure of arrays over the nE = sum of phrase lengths entries):
//   D[e]       symbol value          rem[e]   symbols after e inside its phrase (0 for the last symbol)
//   einfo[e]   16-byte record read once by the group stage (left symbol + 1, frequency, valid / full flags)
//   phr_of[e]  phrase of the entry -- only under GRLGPU_FLAG_KEEP_DICT (test hooks)
// Suffix order: ONE radix sort of the valid entries on a packed first key (K symbol codes: 0 = past the
// terminator, 1..A = symbol+1, A+1 = terminator, so a proper prefix compares greater; spare bits = top bits of
// code K+1), then only the groups that are still ambiguous are refined -- by key extension (the next K codes,
// straight from D), or by prefix doubling on position-based ranks when phrases are very long.
#pragma once
#include "util.cuh"
#include "parse_kernels.cuh"

namespace grl {

struct IsSuffix {  // phrase_desc bit-vector of the round (exact_par_phase.cpp:311-312, :443)
    const u8* arr;
    u64 sep;
    bool first;
    __device__ __forceinline__ bool operator()(u64 sym) const { return first ? sym == sep : arr[sym] != 0; }
};

// per distinct phrase: first-occurrence position, true length, frequency
static __global__ void __launch_bounds__(256) dict_meta_kernel(const ulonglong2* __restrict__ table, const u32* __restrict__ occ_slots, u64 d,
                                                               const u32* __restrict__ start_bits, const u32* __restrict__ end_bits, u64 n,
                                                               u64* __restrict__ ph_pos, u32* __restrict__ ph_len, u64* __restrict__ ph_freq) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d) return;
    const ulonglong2 ent = table[occ_slots[i]];
    const u64 pos = ent.x >> 24;
    u64 len = ent.x & HT_LEN_SAT;
    if (len == HT_LEN_SAT) len = phrase_len_bits(start_bits, end_bits, n, pos);
    ph_pos[i] = pos;
    ph_len[i] = (u32)len;
    ph_freq[i] = ent.y;
}

// einfo[e] = { left symbol + 1, phrase frequency | valid << 63 | full << 62 }: everything the group stage needs
// about an entry, in one 16-byte record, so that the pass over the sorted order does a single random gather per
// entry. The first symbol of a phrase has no left symbol; its first word carries instead where the phrase's
// metasymbol goes (table slot, or phrase index in multi-GPU rounds) | is_suffix(last symbol) << 63.
constexpr u64 EI_VALID = 1ULL << 63, EI_FULL = 1ULL << 62, EI_FREQ = (1ULL << 62) - 1, EI_SFX = 1ULL << 63;

// entries of a phrase that take part in the suffix order: all but a last symbol that is not is_suffix (exact_par_phase.cpp:163)
template <class CellT, bool FIRST>
__global__ void __launch_bounds__(256) phrase_vlen_kernel(const CellT* __restrict__ text, const u64* __restrict__ ph_pos, const u32* __restrict__ ph_len, u64 d,
                                                          IsSuffix is_suffix, u32* __restrict__ vlen) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d) return;
    const u32 len = ph_len[i];
    vlen[i] = len - ((len && is_suffix(cell_value<CellT, FIRST>(text[ph_pos[i] + len - 1]))) ? 0u : 1u);
}

// One lane per phrase for the per-phrase reads; the entries of a warp's 32 consecutive phrases are consecutive too, so
// the warp then walks them 32 at a time (lane = entry, owner phrase found by a 5-step search over the lanes' offsets)
// and every store is fully coalesced. With ph_voff (offsets of the phrases among the VALID entries, d + 1 values) the
// kernel also emits the first sort key of every valid entry (K symbol codes of `bits` bits, most significant first:
// 0 = past the end, symbol + 1, term_code = terminator, so that a proper prefix compares greater) and its entry id.
template <class CellT, bool FIRST, class SymT>
__global__ void __launch_bounds__(256) dict_gather_kernel(const CellT* __restrict__ text, const u64* __restrict__ ph_pos, const u32* __restrict__ ph_len,
                                                          const u32* __restrict__ ph_off, const u64* __restrict__ ph_freq,
                                                          const u32* __restrict__ target_slots, u64 d, IsSuffix is_suffix, SymT* __restrict__ D,
                                                          u32* __restrict__ phr_of, u32* __restrict__ rem, ulonglong2* __restrict__ einfo,
                                                          const u32* __restrict__ ph_voff, u64 term_code, int bits, int K, int spare,
                                                          u64* __restrict__ keys, u32* __restrict__ vals) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u32 lane = lane_id();
    const u32 nvalid = __popc(__ballot_sync(0xffffffffu, i < d));  // valid lanes are a prefix of the warp
    if (nvalid == 0) return;
    u64 pos = 0, freq = 0, tgt = 0;
    u32 len = 0, off = 0, voff = 0;
    if (i < d) {
        pos = ph_pos[i]; freq = ph_freq[i]; len = ph_len[i]; off = ph_off[i];
        bool sfx_last;
        if (ph_voff) { voff = ph_voff[i]; sfx_last = ph_voff[i + 1] - voff == len; }
        else sfx_last = len && is_suffix(cell_value<CellT, FIRST>(text[pos + len - 1]));  // :443
        tgt = (target_slots ? (u64)target_slots[i] : i) | (sfx_last ? EI_SFX : 0ULL);
    }
    const u32 base = __shfl_sync(0xffffffffu, off, 0);
    const u32 total = __shfl_sync(0xffffffffu, off + len, nvalid - 1) - base;
    const u32 rel = off - base;
    for (u32 j0 = 0; j0 < total; j0 += 32) {
        const u32 j = j0 + lane;
        u32 q = 0;
#pragma unroll
        for (int s = 16; s; s >>= 1) {
            const u32 cand = q + s;
            const u32 r = __shfl_sync(0xffffffffu, rel, cand & 31);
            if (cand < nvalid && r <= j) q = cand;
        }
        const u64 qpos = __shfl_sync(0xffffffffu, pos, q), qfreq = __shfl_sync(0xffffffffu, freq, q), qtgt = __shfl_sync(0xffffffffu, tgt, q);
        const u32 qlen = __shfl_sync(0xffffffffu, len, q), qrel = __shfl_sync(0xffffffffu, rel, q), qvoff = __shfl_sync(0xffffffffu, voff, q);
        if (j >= total) continue;
        const u32 k = j - qrel, r = qlen - 1 - k;
        const u64 v = cell_value<CellT, FIRST>(text[qpos + k]);
        const u64 left = k ? cell_value<CellT, FIRST>(text[qpos + k - 1]) + 1 : qtgt;
        const bool valid = r > 0 || (qtgt & EI_SFX);  // exact_par_phase.cpp:163
        const u64 e = (u64)base + j;
        D[e] = (SymT)v;
        if (phr_of) phr_of[e] = (u32)(i - lane + q);
        rem[e] = r;
        if (einfo) einfo[e] = make_ulonglong2(left, qfreq | (valid ? EI_VALID : 0ULL) | (k == 0 ? EI_FULL : 0ULL));
        if (ph_voff && valid) {
            u64 key = v + 1;
            for (int t = 1; t <= K; t++) {  // t == K: the bits that are left take the TOP `spare` bits of the next code (order-preserving)
                if (t == K && spare == 0) break;
                u64 code = 0;
                if ((u32)t <= r) code = cell_value<CellT, FIRST>(text[qpos + k + t]) + 1;
                else if ((u32)t == r + 1) code = term_code;
                if (t < K) key = (key << bits) | code;
                else {  // monotone squeeze of code K + 1 into `spare` bits; the terminator keeps a value of its own (all ones)
                    const u64 top = (1ULL << spare) - 1ULL, sq = code >> (bits - spare);
                    key = (key << spare) | (code == term_code ? top : (sq < top ? sq : top - 1ULL));
                }
            }
            keys[(u64)qvoff + k] = key;
            vals[(u64)qvoff + k] = (u32)e;
        }
    }
}

// first sort key: K symbol codes of `bits` bits each, most significant first
template <class SymT>
__global__ void __launch_bounds__(256) sfx_first_key_kernel(const SymT* __restrict__ D, const u32* __restrict__ rem, u64 nE, u64 term_code, int bits, int K,
                                                            u64* __restrict__ keys, u32* __restrict__ vals) {
    const u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nE) return;
    const u32 r = rem[e];
    u64 key = 0;
    for (int t = 0; t < K; t++) {
        u64 code = 0;
        if ((u32)t <= r) code = (u64)D[e + t] + 1;
        else if ((u32)t == r + 1) code = term_code;
        key = (bits == 64) ? code : ((key << bits) | code);
    }
    keys[e] = key;
    vals[e] = (u32)e;
}

// after a sort: 1 where the key differs from its predecessor
static __global__ void __launch_bounds__(256) key_head_flags_kernel(const u64* __restrict__ keys, u64 n, u32* __restrict__ flags) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    flags[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u;
}

// ---- refinement of the unresolved groups only (Larsson-Sadakane style prefix doubling) ----
// During refinement rank[e] is position-based: 1 + the position (in the sorted order) of the head of e's
// group, so refining one group never changes the rank of another. A group is unresolved while it has more
// than one member and the compared prefix (h codes) holds no terminator yet.

// after the first sort: head flags, head bitmap, and bitmap of the positions that belong to unresolved groups
static __global__ void __launch_bounds__(256) first_heads_kernel(const u64* __restrict__ keys, u64 n, int bits, int spare, u64 term_code, u32* __restrict__ flags,
                                                                 u32* __restrict__ head_bits, u32* __restrict__ active_bits) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    bool head = false, active = false;
    if (i < n) {
        const u64 k = keys[i];
        head = i == 0 || keys[i - 1] != k;
        const bool next_head = i + 1 == n || keys[i + 1] != k;
        const u64 last = bits >= 64 ? k : ((k >> spare) & ((1ULL << bits) - 1ULL));  // the K-th (last whole) code
        const u64 top = (1ULL << spare) - 1ULL;
        const bool finished = last == 0 || last == term_code || (spare > 0 && (k & top) == top);  // the key already holds the terminator
        active = !(head && next_head) && !finished;
        flags[i] = head ? 1u : 0u;
    }
    const u32 hb = __ballot_sync(0xffffffffu, head), ab = __ballot_sync(0xffffffffu, active);
    if (lane_id() == 0 && (i >> 5) < ((n + 31) >> 5)) { head_bits[i >> 5] = hb; active_bits[i >> 5] = ab; }
}
// head_pos[dense group id] = position of the group's head (pos == nullptr: the index itself)
static __global__ void __launch_bounds__(256) head_pos_kernel(const u32* __restrict__ flags, const u32* __restrict__ excl, const u32* __restrict__ pos, u64 n,
                                                              u32* __restrict__ head_pos) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n && flags[j]) head_pos[excl[j]] = pos ? pos[j] : (u32)j;
}
static __global__ void __launch_bounds__(256) assign_hrank_kernel(const u32* __restrict__ flags, const u32* __restrict__ excl, const u32* __restrict__ head_pos,
                                                                  const u32* __restrict__ entries, u64 n, u32* __restrict__ hrank) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) hrank[entries[j]] = head_pos[excl[j] + flags[j] - 1] + 1;
}
// (entry, rank) pairs of the first sort, and their L2-local scatter after a partition by the entry's high bits
static __global__ void __launch_bounds__(256) hrank_pairs_kernel(const u32* __restrict__ flags, const u32* __restrict__ excl, const u32* __restrict__ head_pos,
                                                                 const u32* __restrict__ entries, u64 n, u32* __restrict__ keys, u32* __restrict__ vals) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) { keys[j] = entries[j]; vals[j] = head_pos[excl[j] + flags[j] - 1] + 1; }
}
static __global__ void __launch_bounds__(256) scatter_pairs_kernel(const u32* __restrict__ keys, const u32* __restrict__ vals, u64 n, u32* __restrict__ dst) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) dst[keys[j]] = vals[j];
}
static __global__ void __launch_bounds__(256) active_keys_kernel(const u32* __restrict__ apos, const u32* __restrict__ order, const u32* __restrict__ hrank,
                                                                 const u32* __restrict__ rem, u64 nA, u64 h, u32 term_rank, int bits, u64* __restrict__ keys,
                                                                 u32* __restrict__ vals) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nA) return;
    const u32 e = order[apos[j]];
    const u64 r = rem[e];
    u64 second = 0;
    if (h <= r) second = hrank[e + h];
    else if (h == r + 1) second = term_rank;
    keys[j] = ((u64)hrank[e] << bits) | second;
    vals[j] = e;
}
static __global__ void __launch_bounds__(256) refine_writeback_kernel(const u32* __restrict__ apos, const u32* __restrict__ vals, const u32* __restrict__ flags,
                                                                      u64 nA, u32* __restrict__ order, u32* head_bits) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nA) return;
    const u32 i = apos[j];
    order[i] = vals[j];
    if (flags[j]) atomicOr(&head_bits[i >> 5], 1u << (i & 31));
}
static __global__ void __launch_bounds__(256) active_next_kernel(const u32* __restrict__ apos, const u32* __restrict__ vals, const u32* __restrict__ head_bits,
                                                                 const u32* __restrict__ rem, u64 nA, u64 nE, u64 h2, u32* __restrict__ aflag) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nA) return;
    const u64 i = apos[j];
    const bool hd = (head_bits[i >> 5] >> (i & 31)) & 1u;
    const bool nh = i + 1 == nE || ((head_bits[(i + 1) >> 5] >> ((i + 1) & 31)) & 1u);
    aflag[j] = (!(hd && nh) && (u64)rem[vals[j]] + 1 >= h2) ? 1u : 0u;
}
static __global__ void __launch_bounds__(256) compact_apos_kernel(const u32* __restrict__ aflag, const u32* __restrict__ excl, const u32* __restrict__ apos, u64 nA,
                                                                  u32* __restrict__ apos_next) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < nA && aflag[j]) apos_next[excl[j]] = apos[j];
}
// ---- refinement by key extension (no rank array): an unresolved group is split by the K codes that follow the
// `dpt` codes its members already share; every pass is local to the dictionary text, so it also works when the
// suffix entries are partitioned over several GPUs. Used when ceil((longest phrase + 1) / K) passes are few. ----
template <class SymT>
__global__ void __launch_bounds__(256) ext_keys_kernel(const u32* __restrict__ apos, const u32* __restrict__ order, const SymT* __restrict__ D,
                                                       const u32* __restrict__ rem, const u32* __restrict__ head_bits, u64 nA, u64 dpt, u64 term_code, int bits,
                                                       int K, u64* __restrict__ keys, u32* __restrict__ vals, u64* __restrict__ nk, u32* __restrict__ ev,
                                                       u32* __restrict__ gflag) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nA) return;
    const u32 i = apos[j], e = order[i];
    const u64 r = ld_gather4(rem + e);
    u64 key = 0;
    for (int t = 0; t < K; t++) {
        const u64 pos = dpt + (u64)t;
        u64 code = 0;
        if (pos <= r) code = (u64)D[e + pos] + 1;
        else if (pos == r + 1) code = term_code;
        key = (bits >= 64) ? code : ((key << bits) | code);
    }
    if (keys) keys[j] = key;
    nk[j] = key;
    if (vals) vals[j] = (u32)j;
    ev[j] = e;
    gflag[j] = (head_bits[i >> 5] >> (i & 31)) & 1u;
}
// second sort key: index of the (unresolved) group the active element belongs to
// (gid[j] = exclusive count of group heads + own flag - 1, folded in place first so that the random gather reads ONE array)
static __global__ void __launch_bounds__(256) ext_gid_kernel(const u32* __restrict__ gflag, u32* __restrict__ gexcl, u64 nA) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < nA) gexcl[j] = gexcl[j] + gflag[j] - 1;
}
static __global__ void __launch_bounds__(256) ext_group_keys_kernel(const u32* __restrict__ vals, const u32* __restrict__ gid, u64 nA, u64* __restrict__ keys) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q < nA) keys[q] = (u64)ld_gather4(gid + vals[q]);
}
static __global__ void __launch_bounds__(256) ext_heads_kernel(const u32* __restrict__ vals, const u64* __restrict__ gkeys, const u64* __restrict__ nk, u64 nA,
                                                               u32* __restrict__ flags) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nA) return;
    flags[q] = (q == 0 || gkeys[q] != gkeys[q - 1] || nk[vals[q]] != nk[vals[q - 1]]) ? 1u : 0u;
}
static __global__ void __launch_bounds__(256) ext_writeback_kernel(const u32* __restrict__ apos, const u32* __restrict__ vals, const u32* __restrict__ ev,
                                                                   const u32* __restrict__ flags, u64 nA, u32* __restrict__ order, u32* head_bits) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nA) return;
    const u32 i = apos[q];
    order[i] = ev[vals[q]];
    if (flags[q]) atomicOr(&head_bits[i >> 5], 1u << (i & 31));
}
static __global__ void __launch_bounds__(256) ext_next_kernel(const u32* __restrict__ apos, const u32* __restrict__ vals, const u32* __restrict__ ev,
                                                              const u32* __restrict__ head_bits, const u32* __restrict__ rem, u64 nA, u64 nE, u64 dpt_next,
                                                              u32* __restrict__ aflag) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nA) return;
    const u64 i = apos[q];
    const bool hd = (head_bits[i >> 5] >> (i & 31)) & 1u;
    const bool nh = i + 1 == nE || ((head_bits[(i + 1) >> 5] >> ((i + 1) & 31)) & 1u);
    aflag[q] = (!(hd && nh) && (u64)rem[ev[vals[q]]] + 1 >= dpt_next) ? 1u : 0u;
}
// ---- tile-local segmented sort of the active set. The members of an unresolved group are contiguous in the active list
// (gflag marks the first of each group) and most groups are tiny, so instead of two device-wide radix sorts per depth
// (by extension key, then stably by group) a CTA stages a window of the list in shared memory and the thread that owns a
// group's first slot insertion-sorts the group in place (stable). Groups that straddle a window or exceed LS_MAXG members
// are flagged and take the device-wide path (a fraction of a percent of the set).
//   perm[q]  = active index of the element that belongs at slot q        flags[q] = 1 where a (sub)group starts at slot q
constexpr int LS_THREADS = 256, LS_ITEMS = 8, LS_WIN = LS_THREADS * LS_ITEMS, LS_MAXG = 48;
static __global__ void __launch_bounds__(LS_THREADS) ext_local_sort_kernel(const u64* __restrict__ nk, const u32* __restrict__ gflag, u64 nA, u32* __restrict__ perm,
                                                                          u32* __restrict__ flags, u32* __restrict__ lflag) {
    __shared__ u64 s_key[LS_WIN];
    __shared__ unsigned short s_idx[LS_WIN];
    __shared__ u8 s_head[LS_WIN + 1], s_left[LS_WIN];
    __shared__ u32 s_first;
    const u64 w0 = (u64)blockIdx.x * LS_WIN;
    const u32 cnt = (u32)((nA - w0) < (u64)LS_WIN ? (nA - w0) : (u64)LS_WIN);
    if (threadIdx.x == 0) { s_first = cnt; s_head[cnt] = (w0 + cnt < nA) ? (u8)gflag[w0 + cnt] : (u8)1; }
    __syncthreads();
    for (u32 s = threadIdx.x; s < cnt; s += LS_THREADS) {
        s_key[s] = nk[w0 + s];
        s_idx[s] = (unsigned short)s;
        const u32 h = gflag[w0 + s];
        s_head[s] = (u8)h;
        s_left[s] = 0;
        if (h) atomicMin(&s_first, s);
    }
    __syncthreads();
    const u32 first = s_first;
    for (u32 s = threadIdx.x; s < first; s += LS_THREADS) s_left[s] = 1;  // tail of a group that started in an earlier window
    const u32 lo = threadIdx.x * LS_ITEMS, hi = lo + LS_ITEMS < cnt ? lo + LS_ITEMS : cnt;
    for (u32 s = lo; s < hi; s++) {
        if (!s_head[s]) continue;
        u32 e = s + 1;
        while (e < cnt && !s_head[e]) e++;
        const bool complete = e < cnt || s_head[cnt];
        if (!complete || e - s > (u32)LS_MAXG) {
            for (u32 q = s; q < e; q++) s_left[q] = 1;
            continue;
        }
        for (u32 q = s + 1; q < e; q++) {  // stable insertion sort of [s, e) by key
            const u64 k = s_key[q];
            const unsigned short ix = s_idx[q];
            u32 r = q;
            while (r > s && s_key[r - 1] > k) { s_key[r] = s_key[r - 1]; s_idx[r] = s_idx[r - 1]; r--; }
            s_key[r] = k;
            s_idx[r] = ix;
        }
    }
    __syncthreads();
    for (u32 s = threadIdx.x; s < cnt; s += LS_THREADS) {
        const u32 left = s_left[s];
        lflag[w0 + s] = left;
        perm[w0 + s] = (u32)w0 + (left ? s : (u32)s_idx[s]);
        flags[w0 + s] = left ? 0u : ((s_head[s] || s_key[s] != s_key[s - 1]) ? 1u : 0u);
    }
}
// the flagged remainder as a list of its own (keys, group-start flags), and its results merged back
static __global__ void __launch_bounds__(256) ext_left_gather_kernel(const u32* __restrict__ lflag, const u32* __restrict__ lexcl, const u64* __restrict__ nk,
                                                                     const u32* __restrict__ gflag, u64 nA, u32* __restrict__ lpos, u64* __restrict__ lk,
                                                                     u64* __restrict__ lnk, u32* __restrict__ lv, u32* __restrict__ lg) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nA || !lflag[j]) return;
    const u32 k = lexcl[j];
    lpos[k] = (u32)j;
    lk[k] = nk[j];
    lnk[k] = nk[j];
    lv[k] = k;
    lg[k] = gflag[j];
}
static __global__ void __launch_bounds__(256) ext_left_scatter_kernel(const u32* __restrict__ lpos, const u32* __restrict__ lvp, const u32* __restrict__ lf, u64 nL,
                                                                      u32* __restrict__ perm, u32* __restrict__ flags) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nL) return;
    const u32 slot = lpos[k];
    perm[slot] = lpos[lvp[k]];
    flags[slot] = lf[k];
}

// dense variant of ginfo (indexed by group) and the per-entry finalisation done in sorted order: no per-entry rank needed
static __global__ void __launch_bounds__(256) pack_ginfo_dense_kernel(const u32* __restrict__ gcnt, const u32* __restrict__ rflag, const u32* __restrict__ rrank, u64 G,
                                                                      u32* __restrict__ ginfo) {
    const u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < G) ginfo[g] = (rrank[g] << 2) | (((gcnt[g] & 0x7fffffffu) > 1) ? 2u : 0u) | (rflag[g] ? 1u : 0u);
}
// metasymbol of every whole phrase (exact_par_phase.cpp:174-176, :437-444) and is_suffix of the next round (:443): a group
// of equal suffixes holds at most one whole phrase, whose destination group_reduce left in gfull
static __global__ void __launch_bounds__(256) full_apply_kernel(const u32* __restrict__ gcnt, const u32* __restrict__ rflag, const u32* __restrict__ rrank,
                                                                const u64* __restrict__ gfull, u64 G, ulonglong2* table, u8* __restrict__ is_suffix_next) {
    const u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G || !rflag[g] || !(gcnt[g] >> 31)) return;
    const u64 r = rrank[g], f = gfull[g];
    table[f >> 2].y = (r << 1) | (f & 1ULL);
    is_suffix_next[r] = (u8)((f >> 1) & 1ULL);
}
// rank marks of the entries of hocc groups (phr_marks + new_phrases_ht, :190-207), pass in sorted order
static __global__ void __launch_bounds__(256) group_apply_kernel(const u32* __restrict__ order, const u32* __restrict__ head_bits, const u32* __restrict__ head_pref,
                                                                 const u32* __restrict__ ginfo, u64 nE, u32* __restrict__ erank) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nE) return;
    const u32 hw = head_bits[i >> 5];
    const u32 g = head_pref[i >> 5] + __popc(hw & (0xffffffffu >> (31 - (i & 31)))) - 1;
    const u32 gi = ginfo[g];
    if ((gi & 3u) != 3u) return;  // only ranked groups with more than one entry
    erank[order[i]] = gi >> 2;
}

// ---- distributed ranking: every rank owns the suffix entries whose first key falls in its range [lo, hi) ----
static __global__ void __launch_bounds__(256) key_sample_kernel(const u64* __restrict__ keys, u64 n, u64 stride, u64 n_samples, u64* __restrict__ out, u32* __restrict__ vals) {
    const u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n_samples) { const u64 i = s * stride; out[s] = keys[i < n ? i : n - 1]; vals[s] = (u32)s; }
}

static __global__ void __launch_bounds__(256) popc_words_kernel(const u32* __restrict__ bits, u64 n_words, u32* __restrict__ cnt) {
    const u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (w < n_words) cnt[w] = __popc(bits[w]);
}

// ---- segmented warp reductions over runs of equal keys that are contiguous across lanes ----
template <class T, class Op>
__device__ __forceinline__ T seg_reduce(T v, u32 seg_last, Op op) {
    const u32 l = lane_id();
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T x = __shfl_down_sync(0xffffffffu, v, o);
        if (l + o <= seg_last) v = op(v, x);
    }
    return v;
}
struct OpSum { template <class T> __device__ __forceinline__ T operator()(T a, T b) const { return a + b; } };
struct OpMin { template <class T> __device__ __forceinline__ T operator()(T a, T b) const { return a < b ? a : b; } };
struct OpMax { template <class T> __device__ __forceinline__ T operator()(T a, T b) const { return a > b ? a : b; } };

// G1: per-group aggregates over the sorted entries (produce_pre_bwt exact_par_phase.cpp:159-187).
// gcnt = entries | full<<31 ; gmin/gmax over (left symbol + 1) of the non-full entries (0 = none).
static __global__ void __launch_bounds__(256) group_reduce_kernel(const u32* __restrict__ order, const u32* __restrict__ head_bits, const u32* __restrict__ head_pref,
                                                                  const ulonglong2* __restrict__ einfo, u64 nE, u32* gcnt, u64* gacc, u64* gmin, u64* gmax,
                                                                  u32* __restrict__ grep, u32* __restrict__ ghead, u64* __restrict__ gfull) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u32 g = 0xffffffffu, cnt = 0;
    u64 acc = 0, mn = ~0ULL, mx = 0;
    bool hd = false, nh = true, is_full = false;
    if (i < nE) {
        const u32 e = order[i];
        const u32 hw = head_bits[i >> 5];
        const u32 upto = hw & (0xffffffffu >> (31 - (i & 31)));  // heads at positions <= i inside the word
        g = head_pref[i >> 5] + __popc(upto) - 1;                // dense group index in sorted order
        hd = (hw >> (i & 31)) & 1u;
        nh = i + 1 == nE || ((head_bits[(i + 1) >> 5] >> ((i + 1) & 31)) & 1u);
        const ulonglong2 ei = ld_gather16(einfo + e);
        if (ei.y & EI_VALID) {
            is_full = (ei.y & EI_FULL) != 0;
            cnt = 1u | (is_full ? 0x80000000u : 0u);
            acc = ei.y & EI_FREQ;
            if (is_full) gfull[g] = ((ei.x & ~EI_SFX) << 2) | ((ei.x >> 63) << 1) | (acc > 1 ? 1ULL : 0ULL);  // at most one per group
            else if (ei.x) mn = mx = ei.x;
        }
        if (hd) { grep[g] = e; ghead[g] = (u32)i; }  // entries keep their position-based rank = head position + 1
    }
    const u32 m = __match_any_sync(0xffffffffu, g);
    const u32 first = __ffs(m) - 1, last = 31 - __clz(m);
    cnt = seg_reduce(cnt, last, OpSum());
    acc = seg_reduce(acc, last, OpSum());
    mn = seg_reduce(mn, last, OpMin());
    mx = seg_reduce(mx, last, OpMax());
    // a group that starts and ends inside this warp is stored directly (consecutive groups -> consecutive
    // addresses); only groups that straddle warps accumulate with atomics on the zero-initialised arrays
    const bool whole = __shfl_sync(0xffffffffu, hd, first) && __shfl_sync(0xffffffffu, nh, last);
    if (lane_id() == first && g != 0xffffffffu && (cnt & 0x7fffffffu)) {
        if (whole) {
            gcnt[g] = cnt;
            gacc[g] = acc;
            if (mx) { gmin[g] = mn; gmax[g] = mx; }
        } else {
            atomicAdd(&gcnt[g], cnt);
            atomicAdd(&gacc[g], acc);
            if (mx) { atomicMin(&gmin[g], mn); atomicMax(&gmax[g], mx); }
        }
    }
}

// G2: ranked / valid flags and the preliminary-BWT symbol of each group (exact_par_phase.cpp:187-216)
static __global__ void __launch_bounds__(256) group_finalize_kernel(const u32* __restrict__ gcnt, const u64* __restrict__ gmin, const u64* __restrict__ gmax, u64 G,
                                                                    u64 bwt_dummy, u64 hocc_dummy, u32* __restrict__ rflag, u32* __restrict__ vflag,
                                                                    u64* __restrict__ psym) {
    const u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    const u32 c = gcnt[g], cnt = c & 0x7fffffffu;
    const bool full = c >> 31, valid = cnt > 0;
    const bool ranked = valid && (full || gmin[g] != gmax[g]);
    rflag[g] = ranked;
    vflag[g] = valid;
    psym[g] = ranked ? (cnt > 1 ? hocc_dummy : bwt_dummy) : (valid ? gmin[g] - 1 : 0);
}

static __global__ void __launch_bounds__(256) prebwt_compact_kernel(const u32* __restrict__ vflag, const u32* __restrict__ vidx, const u64* __restrict__ psym,
                                                                    const u64* __restrict__ gacc, u64 G, u64* __restrict__ csym, u64* __restrict__ clen) {
    const u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G || !vflag[g]) return;
    csym[vidx[g]] = psym[g];
    clen[vidx[g]] = gacc[g];
}

// maximal runs of the compacted (symbol, length) sequence: run id = inclusive count of heads - 1
template <class SymT>
__global__ void __launch_bounds__(256) prebwt_runs_kernel(const u64* __restrict__ csym, const u64* __restrict__ clen, const u32* __restrict__ hflag,
                                                          const u32* __restrict__ hexcl, u64 nV, SymT* __restrict__ run_sym, u64* run_len) {
    const u64 v = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u32 rid = 0xffffffffu;
    u64 len = 0;
    if (v < nV) {
        rid = hexcl[v] + hflag[v] - 1;
        len = clen[v];
        if (hflag[v]) run_sym[rid] = (SymT)csym[v];
    }
    const u32 m = __match_any_sync(0xffffffffu, rid);
    const u32 first = __ffs(m) - 1, last = 31 - __clz(m);
    len = seg_reduce(len, last, OpSum());
    if (lane_id() == first && rid != 0xffffffffu) atomicAdd(&run_len[rid], len);
}

// G4 (prefix-doubling fallback): rank marks of entries in hocc groups (phr_marks + new_phrases_ht, :190-207)
// ginfo_pos[head position of the group] = rank << 2 | hocc << 1 | ranked : entries reach it through their
// position-based rank, so the sorted pass never has to scatter a dense group id back to the entries
static __global__ void __launch_bounds__(256) pack_ginfo_kernel(const u32* __restrict__ gcnt, const u32* __restrict__ rflag, const u32* __restrict__ rrank,
                                                                const u32* __restrict__ ghead, u64 G, u32* __restrict__ ginfo_pos) {
    const u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < G) ginfo_pos[ghead[g]] = (rrank[g] << 2) | (((gcnt[g] & 0x7fffffffu) > 1) ? 2u : 0u) | (rflag[g] ? 1u : 0u);
}
static __global__ void __launch_bounds__(256) entry_finalize_kernel(const u32* __restrict__ rank, u64 nE, const u32* __restrict__ ginfo_pos, u32* __restrict__ erank) {
    const u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nE) return;
    const u32 gi = ginfo_pos[rank[e] - 1];  // rank[e] - 1 = position of the head of e's group in the sorted order
    if ((gi & 3u) == 3u) erank[e] = gi >> 2;
}

// G5: grammar rule of every ranked group from its representative entry (produce_grammar exact_par_phase.cpp:33-87)
template <class SymT>
__global__ void __launch_bounds__(256) rules_kernel(const u32* __restrict__ gcnt, const u32* __restrict__ rflag, const u32* __restrict__ rrank,
                                                    const u32* __restrict__ grep, u64 G, const SymT* __restrict__ D, const u32* __restrict__ rem,
                                                    const u32* __restrict__ erank, IsSuffix is_suffix, u64 alph3, u64 metasym_dummy,
                                                    SymT* __restrict__ rule_l, SymT* __restrict__ rule_r, u8* __restrict__ has_hocc) {
    const u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G || !rflag[g]) return;
    const u32 u = rrank[g];
    has_hocc[u] = (gcnt[g] & 0x7fffffffu) > 1;
    u32 pos = grep[g];
    if (ld_gather(rem + pos) == 0) {  // :38-41 one-symbol suffix
        rule_l[u] = (SymT)metasym_dummy;
        rule_r[u] = ld_gather(D + pos);
        return;
    }
    pos++;
    u32 er = ld_gather(erank + pos);
    while (er == 0xffffffffu && ld_gather(rem + pos) != 0) { pos++; er = ld_gather(erank + pos); }  // :43-44
    const SymT l_sym = ld_gather(D + pos - 1);
    if (er != 0xffffffffu) {  // :49-80
        rule_l[u] = l_sym;
        rule_r[u] = (SymT)(alph3 + er);
    } else {  // :81-85
        const SymT r_sym = ld_gather(D + pos);
        rule_l[u] = (SymT)metasym_dummy;
        rule_r[u] = is_suffix((u64)r_sym) ? r_sym : l_sym;
    }
}

}  // namespace grl
