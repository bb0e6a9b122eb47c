// Multi-GPU parse round with a PARTITIONED global dictionary (SURVEY.md 8e; replaces the thread fan-out and the serial
// join_thread_phrases of mt_parse_strat_t, include/parsing_strategies.h:244-386, and shards the work of
// suffix_induction / produce_pre_bwt / produce_grammar, exact_LMS_induction.h:94-158, exact_par_phase.cpp:14-242).
// Included by grlgpu.cu inside its anonymous namespace (it reuses Round, the text stages and finish_round).
//
// One rank = one GPU = one shard of WHOLE strings (the reference's own split, parsing_strategies.h:208-214). No rank
// ever holds the global dictionary; per round:
//   L  local boundary scan + dedup                                    -> locally distinct phrases with counts
//   E1 all-to-all-v by PHRASE OWNER (content hash % G)                -> every phrase meets its duplicates on one rank,
//      which sums the counts: the dictionary is partitioned by owner (phrase + global frequency + "ends a string" bit)
//   D  every owner lists the suffix entries of its phrases with their packed first key
//   E2 all-to-all-v by KEY RANGE (splitters from an all-gathered sample) of 28-36 byte records {key, left symbol,
//      frequency|flags, entry id, remaining length}: equal suffixes meet on one rank, ranges are in global order
//   O  local radix sort + refinement of ambiguous groups; the next key words of the few entries that need them are
//      asked from their owners (request / reply all-to-all-v per pass, active set only)
//   G  groups, ranked / hocc flags, preliminary-BWT runs of the range; rank offsets from an all-gather of G counts
//   E3 reverse of E2: one 8-byte code per entry (global rank | hocc | representative)
//   U  owners derive the metasymbol of each phrase (code of its first entry) and the grammar rule of every group they
//      hold the representative of (the scan over the following entries of the phrase needs only the owner's codes)
//   E4 all-to-all-v of the rules by RANK RANGE -> every rank holds a dense slice of dict_lev_k in rank order
//   E5 reverse of E1: metasymbols back to the ranks that saw the phrases -> local rewrite
// Per-rank traffic of every collective shrinks as 1/G of the dictionary; what is all-gathered is O(G) scalars and a
// 4096-key sample per rank. "is_suffix" (phrase_desc, exact_par_phase.cpp:311-312,:443) needs no global array here:
// a symbol is_suffix iff it ends a string, so the bit travels with the phrase (end bitmap of the shard).
#pragma once

constexpr u32 MG_FIN = 0x80000000u;    // top bit of a packed phrase length: the phrase ends a string
constexpr u64 MG_NSAMP = 4096;          // first-key samples per rank for the splitters

// ---------------------------------------------------------------- kernels
template <class CellT>
__global__ void __launch_bounds__(256) mg2_pack_kernel(const CellT* __restrict__ text, const u64* __restrict__ ph_pos, const u32* __restrict__ ph_len,
                                                       const u64* __restrict__ ph_cnt, const u32* __restrict__ perm, const u64* __restrict__ offs,
                                                       const u32* __restrict__ end_bits, u64 m, u32* __restrict__ out_lens, u64* __restrict__ out_counts,
                                                       CellT* __restrict__ out_cells) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const u32 i = perm[k];
    const u32 len = ph_len[i];
    const u64 pos = ph_pos[i], o = offs[k], last = pos + len - 1;
    const u32 fin = (end_bits[last >> 5] >> (last & 31)) & 1u;
    out_lens[k] = len | (fin ? MG_FIN : 0u);
    out_counts[k] = ph_cnt[i];
    for (u32 t = 0; t < len; t++) out_cells[o + t] = text[pos + t];
}
static __global__ void __launch_bounds__(256) mg2_strip_fin_kernel(u32* __restrict__ lens, u64 m, u8* __restrict__ fin) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < m) { const u32 v = lens[k]; fin[k] = (u8)(v >> 31); lens[k] = v & ~MG_FIN; }
}
static __global__ void __launch_bounds__(256) mg2_part_fin_kernel(const u32* __restrict__ dense, const u8* __restrict__ fin, u64 m, u8* __restrict__ p_fin) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < m) p_fin[dense[k]] = fin[k];  // every copy of a phrase carries the same bit
}
static __global__ void __launch_bounds__(256) mg2_vlen_kernel(const u32* __restrict__ ph_len, const u8* __restrict__ p_fin, u64 d, u32* __restrict__ vlen) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < d) vlen[i] = ph_len[i] - (p_fin[i] ? 0u : 1u);  // exact_par_phase.cpp:163: a last symbol takes part only if it is_suffix
}
static __global__ void __launch_bounds__(256) mg2_iota_kernel(u32* __restrict__ v, u64 n) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = (u32)i;
}
// destination rank of a key: number of splitters <= key (splitters ascending, n_split = G - 1)
static __global__ void __launch_bounds__(256) mg2_key_dest_kernel(const u64* __restrict__ keys, u64 n, const u64* __restrict__ split, int n_split,
                                                                  u32* __restrict__ dest, u32* __restrict__ idx) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const u64 k = keys[j];
    u32 g = 0;
    for (int s = 0; s < n_split; s++) g += split[s] <= k ? 1u : 0u;
    dest[j] = g;
    idx[j] = (u32)j;
}
// first[g] = number of sorted keys < g, g = 0..n_vals (one thread per g)
template <class KeyT>
__global__ void mg2_bounds_kernel(const KeyT* __restrict__ keys, u64 m, u32 n_vals, u64* __restrict__ first) {
    const u32 g = threadIdx.x;
    if (g > n_vals) return;
    u64 lo = 0, hi = m;
    while (lo < hi) {
        const u64 mid = (lo + hi) >> 1;
        if ((u64)keys[mid] < (u64)g) lo = mid + 1; else hi = mid;
    }
    first[g] = lo;
}
// the record of every valid entry, written in destination order (q-th record = valid entry perm[q])
// YT: the frequency word travels in 32 bits (frequency | full << 31) whenever the round's highest frequency is below 2^30
template <class SymT, class YT>
__global__ void __launch_bounds__(256) mg2_build_send_kernel(const u32* __restrict__ pos, u64 nS, const u64* __restrict__ keys, const u32* __restrict__ vals,
                                                             const SymT* __restrict__ D, const u32* __restrict__ rem, const u32* __restrict__ phr_of,
                                                             const u32* __restrict__ ph_off, const u64* __restrict__ ph_freq, u64* __restrict__ o_key,
                                                             SymT* __restrict__ o_left, YT* __restrict__ o_y, u32* __restrict__ o_id, u32* __restrict__ o_rem) {
    // source order: keys, entry ids and everything they index are read front to back; the writes form one ascending stream per
    // destination (gathering through the partition's permutation instead re-reads every sector once per destination)
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nS) return;
    const u32 q = pos[j], e = vals[j], i = phr_of[e];
    const bool full = e == ph_off[i];
    o_key[q] = keys[j];
    o_left[q] = full ? (SymT)0 : (SymT)(D[e - 1] + 1);  // left symbol + 1; a whole phrase has none
    if constexpr (sizeof(YT) == 4) o_y[q] = (YT)((u32)ph_freq[i] | (full ? 0x80000000u : 0u));
    else o_y[q] = (YT)(ph_freq[i] | EI_VALID | (full ? EI_FULL : 0ULL));
    o_id[q] = e;
    o_rem[q] = rem[e];
}
// pos[perm[q]] = q: where the partition put every source item
static __global__ void __launch_bounds__(256) mg2_invert_perm_kernel(const u32* __restrict__ perm, u64 n, u32* __restrict__ pos) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q < n) pos[perm[q]] = (u32)q;
}
// ---- distributed key extension: the active items ask the owners of their entries for the next K codes ----
// source rank of a received item = segment of the receive buffer it lies in (seg_off: G + 1 ascending offsets)
static __global__ void __launch_bounds__(256) mg2_ext_req_kernel(const u32* __restrict__ apos, const u32* __restrict__ order, const u64* __restrict__ seg_off, int G,
                                                                 const u32* __restrict__ head_bits, u64 nA, u32* __restrict__ src, u32* __restrict__ idx,
                                                                 u32* __restrict__ gflag) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nA) return;
    const u32 i = apos[j], item = order[i];
    u32 s = 0;
    for (int g = 1; g < G; g++) s += seg_off[g] <= (u64)item ? 1u : 0u;
    src[j] = s;
    idx[j] = (u32)j;
    gflag[j] = (head_bits[i >> 5] >> (i & 31)) & 1u;
}
static __global__ void __launch_bounds__(256) mg2_ext_req_ids_kernel(const u32* __restrict__ perm_j, const u32* __restrict__ apos, const u32* __restrict__ order,
                                                                     const u32* __restrict__ r_id, u64 nA, u32* __restrict__ req_ids) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q < nA) req_ids[q] = r_id[order[apos[perm_j[q]]]];
}
template <class SymT>
__global__ void __launch_bounds__(256) mg2_ext_keys_owner_kernel(const SymT* __restrict__ D, const u32* __restrict__ rem, const u32* __restrict__ ids, u64 m, u64 dpt,
                                                                 u64 term_code, int bits, int K, u64* __restrict__ keys) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    const u32 e = ids[q];
    const u64 r = rem[e];
    u64 key = 0;
    for (int t = 0; t < K; t++) {
        const u64 pos = dpt + (u64)t;
        u64 code = 0;
        if (pos <= r) code = (u64)D[(u64)e + pos] + 1;
        else if (pos == r + 1) code = term_code;
        key = (bits >= 64) ? code : ((key << bits) | code);
    }
    keys[q] = key;
}
static __global__ void __launch_bounds__(256) mg2_ext_scatter_kernel(const u32* __restrict__ perm_j, const u64* __restrict__ resp, const u32* __restrict__ apos,
                                                                     const u32* __restrict__ order, u64 nA, u64* __restrict__ keys, u64* __restrict__ nk,
                                                                     u32* __restrict__ vals, u32* __restrict__ ev) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nA) return;
    const u32 j = perm_j[q];
    const u64 k = resp[q];
    if (keys) keys[j] = k;
    nk[j] = k;
    if (vals) vals[j] = j;
    ev[j] = order[apos[j]];
}
// the two record fields the group stage reads, side by side: ONE random 16-byte gather per entry instead of two
template <class SymT, class YT>
__global__ void __launch_bounds__(256) mg2_zip_kernel(const SymT* __restrict__ r_left, const YT* __restrict__ r_y, u64 nL, ulonglong2* __restrict__ ei) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nL) return;
    u64 y;
    if constexpr (sizeof(YT) == 4) { const u32 v = (u32)r_y[i]; y = (u64)(v & 0x7fffffffu) | EI_VALID | ((v >> 31) ? EI_FULL : 0ULL); }
    else y = (u64)r_y[i];
    ei[i] = make_ulonglong2((u64)r_left[i], y);
}
// group aggregates over the sorted items of this range (produce_pre_bwt exact_par_phase.cpp:159-187)
static __global__ void __launch_bounds__(256) mg2_group_reduce_kernel(const u32* __restrict__ order, const u32* __restrict__ head_bits, const u32* __restrict__ head_pref,
                                                                     const ulonglong2* __restrict__ r_ei, u64 nL, u32* gcnt, u64* gacc, u64* gmin, u64* gmax) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u32 g = 0xffffffffu, cnt = 0;
    u64 acc = 0, mn = ~0ULL, mx = 0;
    bool hd = false, nh = true;
    if (i < nL) {
        const u32 it = order[i];
        const u32 hw = head_bits[i >> 5];
        g = head_pref[i >> 5] + __popc(hw & (0xffffffffu >> (31 - (i & 31)))) - 1;
        hd = (hw >> (i & 31)) & 1u;
        nh = i + 1 == nL || ((head_bits[(i + 1) >> 5] >> ((i + 1) & 31)) & 1u);
        const ulonglong2 ei = ld_gather16(r_ei + it);
        const bool is_full = (ei.y & EI_FULL) != 0;
        cnt = 1u | (is_full ? 0x80000000u : 0u);
        acc = ei.y & EI_FREQ;
        if (!is_full && ei.x) mn = mx = ei.x;
    }
    const u32 m = __match_any_sync(0xffffffffu, g);
    const u32 first = __ffs(m) - 1, last = 31 - __clz(m);
    cnt = seg_reduce(cnt, last, OpSum());
    acc = seg_reduce(acc, last, OpSum());
    mn = seg_reduce(mn, last, OpMin());
    mx = seg_reduce(mx, last, OpMax());
    const bool whole = __shfl_sync(0xffffffffu, hd, first) && __shfl_sync(0xffffffffu, nh, last);
    if (lane_id() == first && g != 0xffffffffu) {
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
// code of every item, at the item's position in the receive buffer: 0 = its group is not ranked, else
// ((global rank << 2) | hocc << 1 | representative) + 1   (phr_marks / new_phrases_ht, exact_par_phase.cpp:190-207)
template <class CodeT>
__global__ void __launch_bounds__(256) mg2_codes_kernel(const u32* __restrict__ order, const u32* __restrict__ head_bits, const u32* __restrict__ head_pref,
                                                        const u32* __restrict__ ginfo, u64 nL, u64 rank_base, CodeT* __restrict__ codes) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nL) return;
    const u32 hw = head_bits[i >> 5];
    const u32 g = head_pref[i >> 5] + __popc(hw & (0xffffffffu >> (31 - (i & 31)))) - 1;
    const u32 gi = ginfo[g];
    const u64 rep = (hw >> (i & 31)) & 1u;
    if (gi & 1u) codes[order[i]] = (CodeT)(((((u64)(gi >> 2) + rank_base) << 2) | (u64)(gi & 2u) | rep) + 1ULL);  // (zero-initialised: unranked groups cost no scattered write)
}
template <class CodeT>
__global__ void __launch_bounds__(256) mg2_codes_to_entries_kernel(const u32* __restrict__ vals, const u32* __restrict__ pos, const CodeT* __restrict__ back, u64 nS,
                                                                   u64* __restrict__ ecode) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;   // source order again: ascending entry ids, one ascending read stream per destination
    if (j < nS) ecode[vals[j]] = (u64)back[pos[j]];
}
// metasymbol of every phrase of the partition: rank of the group of its first entry (a whole phrase is always ranked)
static __global__ void __launch_bounds__(256) mg2_meta_kernel(const u64* __restrict__ ecode, const u32* __restrict__ ph_off, const u64* __restrict__ ph_freq, u64 d,
                                                              u64* __restrict__ p_meta, u32* err) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d) return;
    const u64 c = ecode[ph_off[i]];
    if (!c) { atomicExch(err, 1u); return; }
    p_meta[i] = (((c - 1) >> 2) << 1) | (ph_freq[i] > 1 ? 1ULL : 0ULL);  // exact_par_phase.cpp:174-176
}
static __global__ void __launch_bounds__(256) mg2_rule_flags_kernel(const u64* __restrict__ ecode, u64 nE, u32* __restrict__ flags) {
    const u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < nE) { const u64 c = ecode[e]; flags[e] = (c && ((c - 1) & 1ULL)) ? 1u : 0u; }
}
// grammar rule of every group whose representative entry lives here (produce_grammar exact_par_phase.cpp:33-87)
template <class SymT>
__global__ void __launch_bounds__(256) mg2_rules_kernel(const u64* __restrict__ ecode, const SymT* __restrict__ D, const u32* __restrict__ rem,
                                                        const u32* __restrict__ phr_of, const u8* __restrict__ p_fin, const u32* __restrict__ flags,
                                                        const u32* __restrict__ excl, u64 nE, u64 alph3, u64 metasym_dummy, u64* __restrict__ o_u,
                                                        SymT* __restrict__ o_l, SymT* __restrict__ o_r, u8* __restrict__ o_h, uint4* __restrict__ o_rec,
                                                        u32* __restrict__ o_key32) {
    const u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nE || !flags[e]) return;
    const u32 k = excl[e];
    const u64 c = ecode[e] - 1;
    SymT l, r;
    u64 pos = e;
    if (rem[pos] == 0) {  // :38-41 one-symbol suffix
        l = (SymT)metasym_dummy;
        r = D[pos];
    } else {
        pos++;
        u64 cc = ecode[pos];
        bool hocc = cc && ((cc - 1) & 2ULL);
        while (!hocc && rem[pos] != 0) { pos++; cc = ecode[pos]; hocc = cc && ((cc - 1) & 2ULL); }  // :43-44
        const SymT l_sym = D[pos - 1];
        if (hocc) {  // :49-80
            l = l_sym;
            r = (SymT)(alph3 + ((cc - 1) >> 2));
        } else {  // :81-85: pos is the phrase's last symbol, which is_suffix iff the phrase ends a string
            const SymT r_sym = D[pos];
            l = (SymT)metasym_dummy;
            r = p_fin[phr_of[pos]] ? r_sym : l_sym;
        }
    }
    if (o_rec) {  // 32-bit symbols and ranks: one 16-byte record per rule, so the gather that follows the sort costs one sector, not four
        o_rec[k] = make_uint4((u32)(c >> 2), (u32)l, (u32)r, (u32)((c >> 1) & 1ULL));
        o_key32[k] = (u32)(c >> 2);
    } else {
        o_u[k] = c >> 2;
        o_h[k] = (u8)((c >> 1) & 1ULL);
        o_l[k] = l;
        o_r[k] = r;
    }
}
// the rules of this rank sorted by their (global) rank: first[g] = number of them below bases[g], g = 0..G (one thread per g):
// the owner of a rank is the range it falls in, so the sorted list is already grouped by destination
template <class KeyT>
__global__ void mg2_rule_bounds_kernel(const KeyT* __restrict__ sorted_u, u64 n, const u64* __restrict__ bases, int G, u64* __restrict__ first) {
    const int g = threadIdx.x;
    if (g > G) return;
    if (g == G) { first[g] = n; return; }
    const u64 b = bases[g];
    u64 lo = 0, hi = n;
    while (lo < hi) {
        const u64 mid = (lo + hi) >> 1;
        if ((u64)sorted_u[mid] < b) lo = mid + 1; else hi = mid;
    }
    first[g] = lo;
}
// UT: the rank travels in 32 bits whenever the round hands out fewer than 2^32 ranks
template <class SymT, class UT>
__global__ void __launch_bounds__(256) mg2_rule_send_kernel(const u32* __restrict__ perm, u64 n, const u64* __restrict__ u, const SymT* __restrict__ l,
                                                            const SymT* __restrict__ r, const u8* __restrict__ h, UT* __restrict__ su, SymT* __restrict__ sl,
                                                            SymT* __restrict__ sr, u8* __restrict__ sh) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const u32 k = perm[q];
    su[q] = (UT)u[k]; sl[q] = l[k]; sr[q] = r[k]; sh[q] = h[k];
}
static __global__ void __launch_bounds__(256) mg2_rule_send_rec_kernel(const u32* __restrict__ perm, u64 n, const uint4* __restrict__ rec, u32* __restrict__ su,
                                                                       u32* __restrict__ sl, u32* __restrict__ sr, u8* __restrict__ sh) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const ulonglong2 v = ld_gather16(reinterpret_cast<const ulonglong2*>(rec) + perm[q]);
    su[q] = (u32)v.x; sl[q] = (u32)(v.x >> 32); sr[q] = (u32)v.y; sh[q] = (u8)(v.y >> 32);
}
template <class SymT, class UT>
__global__ void __launch_bounds__(256) mg2_rule_scatter_kernel(const UT* __restrict__ u, const SymT* __restrict__ l, const SymT* __restrict__ r,
                                                               const u8* __restrict__ h, u64 m, u64 base, u64 tot_local, SymT* __restrict__ rule_l,
                                                               SymT* __restrict__ rule_r, u8* __restrict__ has_hocc, u32* err) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    const u64 k = (u64)u[q] - base;
    if (k >= tot_local) { atomicExch(err, 1u); return; }
    rule_l[k] = l[q]; rule_r[k] = r[q]; has_hocc[k] = h[q];
}
static __global__ void mg2_add_u64_kernel(u64* p, u64 v) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *p += v;
}

// ---------------------------------------------------------------- host helpers
// GRLGPU_TRACE: wall time of every stage of a multi-GPU round on this rank (a stream synchronisation per lap; off otherwise)
struct Mg2StageClock {
    bool on;
    int rank, round;
    cudaStream_t st;
    std::chrono::steady_clock::time_point t0;
    Mg2StageClock(int rank_, int round_, cudaStream_t st_) : on(getenv("GRLGPU_TRACE") != nullptr), rank(rank_), round(round_), st(st_) {
        if (on) { cudaStreamSynchronize(st); t0 = std::chrono::steady_clock::now(); }
    }
    void lap(const char* what) {
        if (!on) return;
        cudaStreamSynchronize(st);
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[grlgpu] rank %d round %d stage %-22s %8.2f ms\n", rank, round, what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};
inline std::vector<u64> mg2_offsets(const std::vector<u64>& counts, u64 elem_bytes) {
    std::vector<u64> off(counts.size() + 1, 0);
    for (size_t i = 0; i < counts.size(); i++) off[i + 1] = off[i] + counts[i] * elem_bytes;
    return off;
}
inline u64 mg2_sum(const std::vector<u64>& v) { u64 s = 0; for (u64 x : v) s += x; return s; }
// every rank's vector of `k` u64 values, rank-major
inline std::vector<u64> mg2_gather(Comm& cm, const std::vector<u64>& mine, cudaStream_t st) {
    std::vector<u64> all(mine.size() * (size_t)cm.world);
    cm.all_gather_host(mine.data(), mine.size() * sizeof(u64), all.data(), st);
    return all;
}
// my per-peer element counts -> what every peer sends to me (column `me` of the count matrix)
inline std::vector<u64> mg2_exchange_counts(Comm& cm, const std::vector<u64>& send_counts, cudaStream_t st) {
    const std::vector<u64> all = mg2_gather(cm, send_counts, st);
    std::vector<u64> recv((size_t)cm.world);
    for (int p = 0; p < cm.world; p++) recv[(size_t)p] = all[(size_t)p * (size_t)cm.world + (size_t)cm.rank];
    return recv;
}
inline void mg2_a2a_soa(Comm& cm, const std::vector<Comm::SoaPart>& parts, const std::vector<u64>& send_counts, const std::vector<u64>& recv_counts, cudaStream_t st) {
    cm.all_to_all_soa(parts.data(), (int)parts.size(), send_counts.data(), recv_counts.data(), st);
}
template <class T>
inline void mg2_a2a(Comm& cm, const T* d_send, const std::vector<u64>& send_counts, T* d_recv, const std::vector<u64>& recv_counts, cudaStream_t st) {
    const std::vector<u64> so = mg2_offsets(send_counts, sizeof(T)), ro = mg2_offsets(recv_counts, sizeof(T));
    cm.all_to_all_v(d_send, so.data(), d_recv, ro.data(), st);
}
// stable partition of (dest, idx) pairs by dest (< 256); returns the permutation in `perm` and the per-destination counts
inline std::vector<u64> mg2_partition(DevBuf<u32>& dest, DevBuf<u32>& idx, u64 n, int G, DevBuf<u32>& perm, cudaStream_t st) {
    std::vector<u64> cnt((size_t)G, 0);
    if (n == 0) { perm.alloc(0, st); return cnt; }
    DevBuf<u32> k2(n, st), v2(n, st);
    u32 *k1 = dest.p, *v1 = idx.p, *ka = k2.p, *va = v2.p;
    radix_partition_u32(&k1, &v1, &ka, &va, n, 0, st);
    DevBuf<u64> first((u64)G + 1, st);
    GRL_LAUNCH("mg_bounds", 0, (mg2_bounds_kernel<u32>), 1, 32, 0, st, k1, n, (u32)G, first.p);
    std::vector<u64> hf((size_t)G + 1);
    d2h_mapped(hf.data(), first.p, ((size_t)G + 1) * 8, st);  // (not a copy-engine job: it would queue behind the asynchronous level copies)
    for (int g = 0; g < G; g++) cnt[(size_t)g] = hf[(size_t)g + 1] - hf[(size_t)g];
    if (v1 == idx.p) perm = std::move(idx); else perm = std::move(v2);
    return cnt;
}

struct Mg2Part {   // this rank's partition of the round's dictionary + what the ranking stage needs from it
    Round PR;
    DevBuf<u8> p_fin;
    DevBuf<u64> p_meta;
    int sym_bits = 0, K = 1, spare = 0;
    u64 max_len_g = 0, max_freq_g = 0;
    explicit Mg2Part(grlgpu_ctx* c) : PR(c) {}
};

template <class CellT, bool FIRST, class SymT>
void mg2_gather(grlgpu_ctx* c, Mg2Part& P) {
    Round& PR = P.PR;
    cudaStream_t st = c->st;
    DevBuf<u32> voff(PR.d + 1, st);
    GRL_LAUNCH("mg_vlen", PR.d * 9, mg2_vlen_kernel, grid_for(PR.d, 256), 256, 0, st, PR.ph_len.p, P.p_fin.p, PR.d, voff.p);
    exclusive_scan<u32, u32>(voff.p, voff.p, PR.d, voff.p + PR.d, st);
    PR.nS = d2h_scalar(voff.p + PR.d, st);
    PR.keys.alloc(PR.nS, st);
    PR.vals.alloc(PR.nS, st);
    PR.D_raw.alloc((PR.nE + 1) * sizeof(SymT), st);
    PR.phr_of.alloc(PR.nE, st);
    PR.rem.alloc(PR.nE, st);
    IsSuffix isuf{nullptr, c->sep, true};  // unused: with ph_voff the kernel derives validity from the offsets
    GRL_LAUNCH("dict_gather", PR.nE * (sizeof(CellT) + sizeof(SymT) + 8) + PR.nS * 12 + PR.d * 32, (dict_gather_kernel<CellT, FIRST, SymT>), grid_for(PR.d, 256), 256, 0, st,
               (const CellT*)PR.dict_text, PR.ph_pos.p, PR.ph_len.p, PR.ph_off.p, PR.ph_freq.p, (const u32*)nullptr, PR.d, isuf, (SymT*)PR.D_raw.p, PR.phr_of.p, PR.rem.p,
               (ulonglong2*)nullptr, (const u32*)voff.p, c->alphabet + 1, P.sym_bits, P.K, P.spare, PR.keys.p, PR.vals.p);
}

// ranking of the partitioned dictionary (steps S..E4 of the header comment); fills c->mg_sl and P.p_meta
template <class SymT>
void mg2_rank(grlgpu_ctx* c, Comm& cm, Mg2Part& P, Mg2Slices& S) {
    const int G = cm.world, me = cm.rank;
    cudaStream_t st = c->st;
    Round& PR = P.PR;
    const u64 A = c->alphabet, nE = PR.nE, nS = PR.nS, d = PR.d;
    const SymT* D = (const SymT*)PR.D_raw.p;
    const int sym_bits = P.sym_bits, K = P.K;
    const int key_bits = std::min(64, sym_bits * K), first_bits = std::min(64, sym_bits * K + P.spare);
    const bool trace = getenv("GRLGPU_TRACE") != nullptr;
    Mg2StageClock clk(me, c->round + 1, st);

    // ---- S: splitters from an all-gathered regular sample of the first keys ----
    std::vector<u64> splitters;
    {
        // ~16 K samples over all ranks put every splitter within about a percent of its quantile; more only lengthens the gather
        const u64 ns_cap = std::min<u64>(MG_NSAMP, std::max<u64>(512, 16384 / (u64)G));
        const u64 ns = std::min<u64>(nS, ns_cap), stride = ns ? std::max<u64>(1, nS / ns) : 1;
        std::vector<u64> mine(ns_cap + 1, 0);
        mine[0] = ns;
        if (ns) {
            DevBuf<u64> sk(ns, st);
            DevBuf<u32> sv(ns, st);
            GRL_LAUNCH("key_sample", 0, key_sample_kernel, grid_for(ns, 256), 256, 0, st, PR.keys.p, nS, stride, ns, sk.p, sv.p);
            d2h_mapped(mine.data() + 1, sk.p, ns * 8, st);
        }
        const std::vector<u64> all = mg2_gather(cm, mine, st);
        std::vector<u64> samp;
        for (int p = 0; p < G; p++) {
            const u64* row = all.data() + (size_t)p * (ns_cap + 1);
            samp.insert(samp.end(), row + 1, row + 1 + row[0]);
        }
        std::sort(samp.begin(), samp.end());
        for (int g = 1; g < G; g++) splitters.push_back(samp.empty() ? 0ULL : samp[(size_t)((u64)g * samp.size() / (u64)G)]);
    }
    clk.lap("S splitters");
    // ---- R: records by key range -> E2 ----
    std::vector<u64> cnt_send, cnt_recv;
    DevBuf<u32> pos;       // slot of the j-th local suffix entry in the send buffers (the codes come back in that order)
    const bool narrow_y = P.max_freq_g < (1ull << 30);  // the records' frequency word fits 32 bits (frequency | full << 31)
    const u64 y_bytes = narrow_y ? 4 : 8;
    DevBuf<u64> r_key;
    DevBuf<u8> r_left_raw, r_y_raw;
    DevBuf<u32> r_id, r_rem;
    u64 nL = 0;
    {
        DevBuf<u64> d_split(std::max<u64>(1, splitters.size()), st);
        if (!splitters.empty()) GRL_CUDA(cudaMemcpyAsync(d_split.p, splitters.data(), splitters.size() * 8, cudaMemcpyHostToDevice, st));
        DevBuf<u32> dest(nS, st), idx(nS, st), perm;
        GRL_LAUNCH("mg_key_dest", nS * 16, mg2_key_dest_kernel, grid_for(nS, 256), 256, 0, st, PR.keys.p, nS, d_split.p, (int)splitters.size(), dest.p, idx.p);
        cnt_send = mg2_partition(dest, idx, nS, G, perm, st);
        dest.release(); idx.release();
        pos.alloc(nS, st);
        if (nS) GRL_LAUNCH("mg_invert_perm", nS * 8, mg2_invert_perm_kernel, grid_for(nS, 256), 256, 0, st, perm.p, nS, pos.p);
        perm.release();
        DevBuf<u64> s_key(nS, st);
        DevBuf<u8> s_left(nS * sizeof(SymT), st), s_y(nS * y_bytes, st);
        DevBuf<u32> s_rem(nS, st), s_id(nS, st);
        if (narrow_y)
            GRL_LAUNCH("mg_build_send", nS * (44 + 2 * sizeof(SymT)), (mg2_build_send_kernel<SymT, u32>), grid_for(nS, 256), 256, 0, st, pos.p, nS, PR.keys.p, PR.vals.p, D, PR.rem.p,
                       PR.phr_of.p, PR.ph_off.p, PR.ph_freq.p, s_key.p, (SymT*)s_left.p, (u32*)s_y.p, s_id.p, s_rem.p);
        else
            GRL_LAUNCH("mg_build_send", nS * (48 + 2 * sizeof(SymT)), (mg2_build_send_kernel<SymT, u64>), grid_for(nS, 256), 256, 0, st, pos.p, nS, PR.keys.p, PR.vals.p, D, PR.rem.p,
                       PR.phr_of.p, PR.ph_off.p, PR.ph_freq.p, s_key.p, (SymT*)s_left.p, (u64*)s_y.p, s_id.p, s_rem.p);
        PR.keys.release();  // PR.vals (entry id of every local suffix entry) stays until the codes are back
        clk.lap("R build records");
        cnt_recv = mg2_exchange_counts(cm, cnt_send, st);
        nL = mg2_sum(cnt_recv);
        if (nL >= 0xfffffff0ull) throw Error(GRLGPU_ERR_LIMIT, "more than 2^32 suffix entries in one rank's key range");
        r_key.alloc(nL, st); r_y_raw.alloc(nL * y_bytes, st); r_left_raw.alloc(nL * sizeof(SymT), st); r_id.alloc(nL, st); r_rem.alloc(nL, st);
        mg2_a2a_soa(cm, {{s_key.p, r_key.p, 8}, {s_left.p, r_left_raw.p, sizeof(SymT)}, {s_y.p, r_y_raw.p, y_bytes}, {s_id.p, r_id.p, 4}, {s_rem.p, r_rem.p, 4}}, cnt_send, cnt_recv,
                    st);
        GRL_CUDA(cudaStreamSynchronize(st));  // the send buffers go back to the pool at the end of this block
    }
    clk.lap("E2 exchange");
    const SymT* r_left = (const SymT*)r_left_raw.p;
    DevBuf<u64> d_seg((u64)G + 1, st);
    {
        const std::vector<u64> seg = mg2_offsets(cnt_recv, 1);
        GRL_CUDA(cudaMemcpyAsync(d_seg.p, seg.data(), seg.size() * 8, cudaMemcpyHostToDevice, st));
        GRL_CUDA(cudaStreamSynchronize(st));
    }
    // ---- O: local order of my range: one sort on the first key, then refinement of the ambiguous groups ----
    const u64 n_words = div_up(std::max<u64>(nL, 1), 32);
    DevBuf<u32> order, head_bits(n_words, st);
    head_bits.zero();
    u64 nA = 0;
    DevBuf<u32> apos;
    {
        DevBuf<u64> keys_alt(nL, st);
        DevBuf<u32> vals(nL, st), vals_alt(nL, st);
        GRL_LAUNCH("mg_iota", nL * 4, mg2_iota_kernel, grid_for(nL, 256), 256, 0, st, vals.p, nL);
        u64 *kp = r_key.p, *ka = keys_alt.p;
        u32 *vp = vals.p, *va = vals_alt.p;
        radix_sort_pairs(&kp, &vp, &ka, &va, nL, first_bits, st);
        if (vp != vals.p) std::swap(vals, vals_alt);
        order = std::move(vals);
        vals_alt.release();
        if (nL) {
            DevBuf<u32> flags(nL, st), active_bits(n_words, st);
            GRL_LAUNCH("first_heads", nL * 12, first_heads_kernel, grid_for(nL, 256), 256, 0, st, kp, nL, sym_bits, P.spare, A + 1, flags.p, head_bits.p, active_bits.p);
            BitmapCompactor ac;
            nA = ac.count(active_bits.p, nL, st);
            apos.alloc(nA, st);
            if (nA) ac.write<u32>(nullptr, apos.p);
        }
        GRL_CUDA(cudaStreamSynchronize(st));
        r_key.release();
    }
    clk.lap("O first-key sort");
    for (u64 dpt = (u64)K;; dpt += (u64)K) {
        // every rank takes part in every pass (it serves key requests even when its own range is resolved)
        u64 nA_max = 0;
        {
            const std::vector<u64> all = mg2_gather(cm, std::vector<u64>{nA}, st);
            for (u64 x : all) nA_max = std::max(nA_max, x);
        }
        if (nA_max == 0) break;
        if (dpt > P.max_len_g + 1) throw Error(GRLGPU_ERR_STATE, "suffix refinement did not converge");
        if (trace) fprintf(stderr, "[grlgpu] rank %d round %d refine: depth %llu, active %llu of %llu\n", me, c->round + 1, dpt, nA, nL);
        DevBuf<u32> gflag(nA, st), perm_j;
        std::vector<u64> req_cnt;
        {
            DevBuf<u32> src(nA, st), idx(nA, st);
            if (nA) GRL_LAUNCH("mg_ext_req", nA * 20, mg2_ext_req_kernel, grid_for(nA, 256), 256, 0, st, apos.p, order.p, d_seg.p, G, head_bits.p, nA, src.p, idx.p, gflag.p);
            req_cnt = mg2_partition(src, idx, nA, G, perm_j, st);
        }
        DevBuf<u32> req_ids(nA, st);
        if (nA) GRL_LAUNCH("mg_ext_req_ids", nA * 20, mg2_ext_req_ids_kernel, grid_for(nA, 256), 256, 0, st, perm_j.p, apos.p, order.p, r_id.p, nA, req_ids.p);
        const std::vector<u64> serve_cnt = mg2_exchange_counts(cm, req_cnt, st);
        const u64 mS = mg2_sum(serve_cnt);
        DevBuf<u32> serve_ids(mS, st);
        mg2_a2a<u32>(cm, req_ids.p, req_cnt, serve_ids.p, serve_cnt, st);
        DevBuf<u64> serve_keys(mS, st), resp(nA, st);
        if (mS) GRL_LAUNCH("mg_ext_keys", mS * 32, (mg2_ext_keys_owner_kernel<SymT>), grid_for(mS, 256), 256, 0, st, D, PR.rem.p, serve_ids.p, mS, dpt, A + 1, sym_bits, K, serve_keys.p);
        mg2_a2a<u64>(cm, serve_keys.p, serve_cnt, resp.p, req_cnt, st);
        GRL_CUDA(cudaStreamSynchronize(st));
        if (nA == 0) continue;
        DevBuf<u64> nk(nA, st);
        DevBuf<u32> ev(nA, st), excl(nA, st), cnt(1, st), perm, flags;
        GRL_LAUNCH("mg_ext_scatter", nA * 40, mg2_ext_scatter_kernel, grid_for(nA, 256), 256, 0, st, perm_j.p, resp.p, apos.p, order.p, nA, (u64*)nullptr, nk.p, (u32*)nullptr, ev.p);
        refine_sort_groups(st, nk.p, gflag.p, nA, key_bits, perm, flags);
        const u32* avp = perm.p;
        GRL_LAUNCH("ext_writeback", nA * 16, ext_writeback_kernel, grid_for(nA, 256), 256, 0, st, apos.p, avp, ev.p, flags.p, nA, order.p, head_bits.p);
        GRL_LAUNCH("ext_next", nA * 16, ext_next_kernel, grid_for(nA, 256), 256, 0, st, apos.p, avp, ev.p, head_bits.p, r_rem.p, nA, nL, dpt + (u64)K, flags.p);
        exclusive_scan<u32, u32>(flags.p, excl.p, nA, cnt.p, st);
        const u64 nA2 = d2h_scalar(cnt.p, st);
        DevBuf<u32> apos2(nA2, st);
        if (nA2) GRL_LAUNCH("compact_apos", nA * 12, compact_apos_kernel, grid_for(nA, 256), 256, 0, st, flags.p, excl.p, apos.p, nA, apos2.p);
        GRL_CUDA(cudaStreamSynchronize(st));
        apos = std::move(apos2);
        nA = nA2;
    }
    apos.release();
    r_id.release(); r_rem.release();
    clk.lap("O refinement");

    // ---- G: groups of my range, ranked / hocc, preliminary BWT of the range ----
    DevBuf<u32> head_pref(n_words, st);
    u64 Gn = 0;
    if (nL) {
        DevBuf<u32> wc(n_words, st), gtot(1, st);
        GRL_LAUNCH("popc_words", n_words * 8, popc_words_kernel, grid_for(n_words, 256), 256, 0, st, head_bits.p, n_words, wc.p);
        exclusive_scan<u32, u32>(wc.p, head_pref.p, n_words, gtot.p, st);
        Gn = d2h_scalar(gtot.p, st);
    }
    DevBuf<u32> gcnt(Gn, st), rflag(Gn, st), vflag(Gn, st), rrank(Gn, st), vidx(Gn, st);
    DevBuf<u64> gacc(Gn, st), gmin(Gn, st), gmax(Gn, st), psym(Gn, st);
    gcnt.zero(); gacc.zero(); gmax.zero(); gmin.fill_ff();
    if (nL) {
        DevBuf<ulonglong2> r_ei(nL, st);
        if (narrow_y) GRL_LAUNCH("mg_zip", nL * (20 + sizeof(SymT)), (mg2_zip_kernel<SymT, u32>), grid_for(nL, 256), 256, 0, st, r_left, (const u32*)r_y_raw.p, nL, r_ei.p);
        else GRL_LAUNCH("mg_zip", nL * (24 + sizeof(SymT)), (mg2_zip_kernel<SymT, u64>), grid_for(nL, 256), 256, 0, st, r_left, (const u64*)r_y_raw.p, nL, r_ei.p);
        GRL_LAUNCH("group_reduce", nL * 24 + Gn * 32, mg2_group_reduce_kernel, grid_for(nL, 256), 256, 0, st, order.p, head_bits.p, head_pref.p, r_ei.p, nL, gcnt.p, gacc.p, gmin.p,
                   gmax.p);
        GRL_CUDA(cudaStreamSynchronize(st));
    }
    r_y_raw.release(); r_left_raw.release();
    const u64 bwt_dummy = A + 1, hocc_dummy = A + 2;  // exact_par_phase.hpp:113-115
    GRL_LAUNCH("group_finalize", 0, group_finalize_kernel, grid_for(Gn, 256), 256, 0, st, gcnt.p, gmin.p, gmax.p, Gn, bwt_dummy, hocc_dummy, rflag.p, vflag.p, psym.p);
    DevBuf<u32> cnt2(2, st);
    exclusive_scan<u32, u32>(rflag.p, rrank.p, Gn, cnt2.p, st);
    exclusive_scan<u32, u32>(vflag.p, vidx.p, Gn, cnt2.p + 1, st);
    u32 hc[2];
    d2h_small(hc, cnt2.p, 8, st);
    const u64 tot_local = hc[0], nV = hc[1];
    if (tot_local >= (1ull << 30)) throw Error(GRLGPU_ERR_LIMIT, "more than 2^30 ranks in one rank's key range");
    u64 n_pre_raw = 0;
    S.lvl.sym_bytes = sizeof(SymT);
    {
        DevBuf<u64> csym(nV, st), clen(nV, st);
        GRL_LAUNCH("prebwt_compact", 0, prebwt_compact_kernel, grid_for(Gn, 256), 256, 0, st, vflag.p, vidx.p, psym.p, gacc.p, Gn, csym.p, clen.p);
        DevBuf<u32> hflag(nV, st), hexcl(nV, st), nrun(1, st);
        GRL_LAUNCH("key_head_flags", 0, key_head_flags_kernel, grid_for(nV, 256), 256, 0, st, csym.p, nV, hflag.p);
        exclusive_scan<u32, u32>(hflag.p, hexcl.p, nV, nrun.p, st);
        n_pre_raw = nV ? d2h_scalar(nrun.p, st) : 0;
        S.lvl.pre_sym.alloc(n_pre_raw * sizeof(SymT), st);
        S.lvl.pre_len.alloc(n_pre_raw, st);
        S.lvl.pre_len.zero();
        GRL_LAUNCH("prebwt_runs", 0, (prebwt_runs_kernel<SymT>), grid_for(nV, 256), 256, 0, st, csym.p, clen.p, hflag.p, hexcl.p, nV, (SymT*)S.lvl.pre_sym.p, S.lvl.pre_len.p);
        GRL_CUDA(cudaStreamSynchronize(st));
    }
    // rank offsets and the seams of the preliminary BWT: equal symbols can only meet where two ranges meet
    std::vector<u64> bases((size_t)G + 1, 0);
    {
        std::vector<u64> mine(5, 0);
        mine[0] = tot_local;
        mine[1] = n_pre_raw;
        if (n_pre_raw) {
            SymT fs, ls;
            d2h_small(&fs, (const SymT*)S.lvl.pre_sym.p, sizeof(SymT), st);
            d2h_small(&ls, (const SymT*)S.lvl.pre_sym.p + (n_pre_raw - 1), sizeof(SymT), st);
            d2h_small(&mine[3], S.lvl.pre_len.p, 8, st);
            mine[2] = (u64)fs;
            mine[4] = (u64)ls;
        }
        const std::vector<u64> all = mg2_gather(cm, mine, st);
        std::vector<u64> drop((size_t)G, 0), add((size_t)G, 0);
        int target = -1;
        u64 open_sym = 0;
        for (int p = 0; p < G; p++) {
            const u64* row = all.data() + (size_t)p * 5;
            bases[(size_t)p + 1] = bases[(size_t)p] + row[0];
            if (row[1] == 0) continue;
            if (target >= 0 && row[2] == open_sym) {  // the range's first run continues the open run of an earlier range
                drop[(size_t)p] = 1;
                add[(size_t)target] += row[3];
                if (row[1] == 1) continue;            // nothing else in this range: the open run stays the same
            }
            target = p;
            open_sym = row[4];
        }
        S.pre_first = 0;
        S.n_pre_global = 0;
        for (int p = 0; p < G; p++) {
            const u64 keep = all[(size_t)p * 5 + 1] - drop[(size_t)p];
            if (p < me) S.pre_first += keep;
            S.n_pre_global += keep;
        }
        S.pre_drop = drop[(size_t)me];
        S.lvl.n_pre = n_pre_raw;
        if (add[(size_t)me]) GRL_LAUNCH("mg_add_u64", 0, mg2_add_u64_kernel, 1, 32, 0, st, S.lvl.pre_len.p + (n_pre_raw - 1), add[(size_t)me]);
    }
    S.rank_base = bases[(size_t)me];
    S.lvl.tot = tot_local;
    S.tot_global = bases[(size_t)G];
    clk.lap("G groups + pre-BWT");
    // ---- E3: one code per entry back to its owner ----
    DevBuf<u64> ecode(nE, st);
    {
        DevBuf<u32> ginfo(Gn, st);
        GRL_LAUNCH("pack_ginfo_dense", Gn * 16, pack_ginfo_dense_kernel, grid_for(Gn, 256), 256, 0, st, gcnt.p, rflag.p, rrank.p, Gn, ginfo.p);
        const bool narrow_code = S.tot_global < (1ull << 29);  // ((rank << 2) | flags) + 1 fits 32 bits
        const u64 cb = narrow_code ? 4 : 8;
        DevBuf<u8> codes(nL * cb, st), back(nS * cb, st);
        codes.zero();
        if (nL) {
            if (narrow_code) GRL_LAUNCH("mg_codes", nL * 20, (mg2_codes_kernel<u32>), grid_for(nL, 256), 256, 0, st, order.p, head_bits.p, head_pref.p, ginfo.p, nL, S.rank_base, (u32*)codes.p);
            else GRL_LAUNCH("mg_codes", nL * 24, (mg2_codes_kernel<u64>), grid_for(nL, 256), 256, 0, st, order.p, head_bits.p, head_pref.p, ginfo.p, nL, S.rank_base, (u64*)codes.p);
        }
        mg2_a2a_soa(cm, {{codes.p, back.p, cb}}, cnt_recv, cnt_send, st);
        ecode.zero();
        if (nS) {
            if (narrow_code) GRL_LAUNCH("mg_codes_to_entries", nS * 20, (mg2_codes_to_entries_kernel<u32>), grid_for(nS, 256), 256, 0, st, PR.vals.p, pos.p, (const u32*)back.p, nS, ecode.p);
            else GRL_LAUNCH("mg_codes_to_entries", nS * 24, (mg2_codes_to_entries_kernel<u64>), grid_for(nS, 256), 256, 0, st, PR.vals.p, pos.p, (const u64*)back.p, nS, ecode.p);
        }
        GRL_CUDA(cudaStreamSynchronize(st));
    }
    order.release(); head_bits.release(); head_pref.release(); pos.release(); PR.vals.release();
    gcnt.release(); rflag.release(); vflag.release(); rrank.release(); vidx.release(); gacc.release(); gmin.release(); gmax.release(); psym.release();
    clk.lap("E3 codes back");
    // ---- U: metasymbols of my phrases, rules of the groups whose representative I own -> E4 by rank range ----
    P.p_meta.alloc(d, st);
    DevBuf<u32> err(1, st);
    err.zero();
    if (d) GRL_LAUNCH("mg_meta", d * 28, mg2_meta_kernel, grid_for(d, 256), 256, 0, st, ecode.p, PR.ph_off.p, PR.ph_freq.p, d, P.p_meta.p, err.p);
    u64 nR = 0;
    DevBuf<u32> rfl(nE, st), rex(nE, st), rc(1, st);
    if (nE) {
        GRL_LAUNCH("mg_rule_flags", nE * 12, mg2_rule_flags_kernel, grid_for(nE, 256), 256, 0, st, ecode.p, nE, rfl.p);
        exclusive_scan<u32, u32>(rfl.p, rex.p, nE, rc.p, st);
        nR = d2h_scalar(rc.p, st);
    }
    const u64 alph3 = A + 3, metasym_dummy = alph3 + S.tot_global + 1;  // exact_par_phase.cpp:19-20
    std::vector<u64> rs_cnt, rr_cnt;
    {
        const bool narrow_u = S.tot_global < (1ull << 32);
        const u64 ub = narrow_u ? 4 : 8;
        const bool zip = narrow_u && sizeof(SymT) == 4;  // 32-bit symbols and ranks: the rules travel through the sort as 16-byte records
        DevBuf<u64> ru(zip ? 0 : nR, st);
        DevBuf<u8> rl(zip ? 0 : nR * sizeof(SymT), st), rr(zip ? 0 : nR * sizeof(SymT), st), rh(zip ? 0 : nR, st);
        DevBuf<uint4> rec(zip ? nR : 0, st);
        DevBuf<u32> k32(zip ? nR : 0, st);
        if (nE) GRL_LAUNCH("rules", nE * 12 + nR * 64, (mg2_rules_kernel<SymT>), grid_for(nE, 256), 256, 0, st, ecode.p, D, PR.rem.p, PR.phr_of.p, P.p_fin.p, rfl.p, rex.p, nE, alph3,
                           metasym_dummy, ru.p, (SymT*)rl.p, (SymT*)rr.p, rh.p, zip ? rec.p : (uint4*)nullptr, k32.p);
        rfl.release(); rex.release();
        DevBuf<u64> d_bases((u64)G + 1, st);
        GRL_CUDA(cudaMemcpyAsync(d_bases.p, bases.data(), ((size_t)G + 1) * 8, cudaMemcpyHostToDevice, st));
        // the rules leave sorted by rank: every destination then receives G ascending streams and its scatter into the rank-ordered
        // slice is nearly sequential (in entry order the ranks are random: one DRAM sector per rule and array)
        DevBuf<u32> perm;
        rs_cnt.assign((size_t)G, 0);
        {
            DevBuf<u64> first((u64)G + 1, st);
            DevBuf<u32> sv(nR, st), sv_alt(nR, st);
            if (nR) GRL_LAUNCH("mg_iota", nR * 4, mg2_iota_kernel, grid_for(nR, 256), 256, 0, st, sv.p, nR);
            u32 *vp = sv.p, *va = sv_alt.p;
            const int rank_bits = std::max(1, bit_width64(S.tot_global));
            if (zip) {
                DevBuf<u32> k32_alt(nR, st);
                u32 *kp = k32.p, *ka = k32_alt.p;
                radix_sort_pairs_u32(&kp, &vp, &ka, &va, nR, rank_bits, st);
                GRL_LAUNCH("mg_rule_bounds", 0, (mg2_rule_bounds_kernel<u32>), 1, 32, 0, st, kp, nR, d_bases.p, G, first.p);
                GRL_CUDA(cudaStreamSynchronize(st));  // k32_alt goes back to the pool
            } else {
                DevBuf<u64> sk(nR, st), sk_alt(nR, st);
                if (nR) GRL_CUDA(cudaMemcpyAsync(sk.p, ru.p, nR * 8, cudaMemcpyDeviceToDevice, st));
                u64 *kp = sk.p, *ka = sk_alt.p;
                radix_sort_pairs(&kp, &vp, &ka, &va, nR, rank_bits, st);
                GRL_LAUNCH("mg_rule_bounds", 0, (mg2_rule_bounds_kernel<u64>), 1, 32, 0, st, kp, nR, d_bases.p, G, first.p);
                GRL_CUDA(cudaStreamSynchronize(st));
            }
            std::vector<u64> hf((size_t)G + 1);
            d2h_mapped(hf.data(), first.p, ((size_t)G + 1) * 8, st);
            for (int g = 0; g < G; g++) rs_cnt[(size_t)g] = hf[(size_t)g + 1] - hf[(size_t)g];
            if (vp != sv.p) std::swap(sv, sv_alt);
            perm = std::move(sv);
        }
        k32.release();
        DevBuf<u8> su(nR * ub, st), sl(nR * sizeof(SymT), st), sr(nR * sizeof(SymT), st), sh(nR, st);
        if (nR) {
            if (zip)
                GRL_LAUNCH("mg_rule_send", nR * (4 + 32 + 13), mg2_rule_send_rec_kernel, grid_for(nR, 256), 256, 0, st, perm.p, nR, rec.p, (u32*)su.p, (u32*)sl.p, (u32*)sr.p, sh.p);
            else if (narrow_u)
                GRL_LAUNCH("mg_rule_send", nR * 2 * (9 + 2 * sizeof(SymT)), (mg2_rule_send_kernel<SymT, u32>), grid_for(nR, 256), 256, 0, st, perm.p, nR, ru.p, (const SymT*)rl.p,
                           (const SymT*)rr.p, rh.p, (u32*)su.p, (SymT*)sl.p, (SymT*)sr.p, sh.p);
            else
                GRL_LAUNCH("mg_rule_send", nR * 2 * (9 + 2 * sizeof(SymT)), (mg2_rule_send_kernel<SymT, u64>), grid_for(nR, 256), 256, 0, st, perm.p, nR, ru.p, (const SymT*)rl.p,
                           (const SymT*)rr.p, rh.p, (u64*)su.p, (SymT*)sl.p, (SymT*)sr.p, sh.p);
        }
        clk.lap("U rules by rank");
        rr_cnt = mg2_exchange_counts(cm, rs_cnt, st);
        const u64 mR = mg2_sum(rr_cnt);
        if (mR != tot_local) throw Error(GRLGPU_ERR_STATE, "multi-GPU round: " + std::to_string(mR) + " rules arrived for " + std::to_string(tot_local) + " ranks of this range");
        DevBuf<u8> qu(mR * ub, st), ql(mR * sizeof(SymT), st), qr(mR * sizeof(SymT), st), qh(mR, st);
        mg2_a2a_soa(cm, {{su.p, qu.p, ub}, {sl.p, ql.p, sizeof(SymT)}, {sr.p, qr.p, sizeof(SymT)}, {sh.p, qh.p, 1}}, rs_cnt, rr_cnt, st);
        S.lvl.rule_l.alloc(tot_local * sizeof(SymT), st);
        S.lvl.rule_r.alloc(tot_local * sizeof(SymT), st);
        S.lvl.has_hocc.alloc(tot_local, st);
        if (mR) {
            if (narrow_u)
                GRL_LAUNCH("mg_rule_scatter", mR * 2 * (9 + 2 * sizeof(SymT)), (mg2_rule_scatter_kernel<SymT, u32>), grid_for(mR, 256), 256, 0, st, (const u32*)qu.p, (const SymT*)ql.p,
                           (const SymT*)qr.p, qh.p, mR, S.rank_base, tot_local, (SymT*)S.lvl.rule_l.p, (SymT*)S.lvl.rule_r.p, S.lvl.has_hocc.p, err.p);
            else
                GRL_LAUNCH("mg_rule_scatter", mR * 2 * (9 + 2 * sizeof(SymT)), (mg2_rule_scatter_kernel<SymT, u64>), grid_for(mR, 256), 256, 0, st, (const u64*)qu.p, (const SymT*)ql.p,
                           (const SymT*)qr.p, qh.p, mR, S.rank_base, tot_local, (SymT*)S.lvl.rule_l.p, (SymT*)S.lvl.rule_r.p, S.lvl.has_hocc.p, err.p);
        }
        if (d2h_scalar(err.p, st)) throw Error(GRLGPU_ERR_STATE, "multi-GPU round: a phrase came back unranked or a rule left its rank range");
    }
    clk.lap("E4 rules exchange");
    S.valid = true;
}

// one multi-GPU parse round on this rank (all ranks call it together)
template <class CellT, bool FIRST>
void mg2_round_t(grlgpu_ctx* c, Comm& cm, grlgpu_round_t* out) {
    const int G = cm.world, me = cm.rank;
    cudaStream_t st = c->st;
    if (G > 31) throw Error(GRLGPU_ERR_ARG, "at most 31 ranks");
    Mg2Slices& S = c->mg_sl;
    S = Mg2Slices();
    const u64 sent0 = cm.bytes_sent;
    Round R(c);
    Timer t_all(st), t_text(st), t_dict(st);
    Mg2StageClock clk(me, c->round + 1, st);
    t_all.start();
    t_text.start();
    // ---- L: this shard ----
    stage_flags<CellT, FIRST>(R);
    stage_dedup<CellT>(R);
    t_text.stop();
    clk.lap("L text pass");
    t_dict.start();
    // owner of every local distinct phrase = content hash % G; pack by owner
    DevBuf<u32> perm;
    std::vector<u64> s_phr((size_t)G), s_cel((size_t)G);
    DevBuf<u32> s_lens(R.d, st);
    DevBuf<u64> s_counts(R.d, st);
    DevBuf<u8> s_cells;
    {
        DevBuf<u64> keys(R.d, st), keys_alt(R.d, st), offs(R.d + 1, st);
        DevBuf<u32> vals(R.d, st), vals_alt(R.d, st);
        GRL_LAUNCH("phrase_owner", 0, (phrase_owner_kernel<CellT>), grid_for(R.d, 256), 256, 0, st, (const CellT*)c->text, R.ph_pos.p, R.ph_len.p, R.d, (u32)G, keys.p, vals.p);
        u64 *kp = keys.p, *ka = keys_alt.p;
        u32 *vp = vals.p, *va = vals_alt.p;
        radix_sort_pairs(&kp, &vp, &ka, &va, R.d, std::max(1, bit_width64((u64)G - 1)), st);
        if (vp != vals.p) std::swap(vals, vals_alt);
        perm = std::move(vals);
        DevBuf<u32> lens_sorted(R.d, st);
        GRL_LAUNCH("gather_u32", 0, gather_u32_kernel, grid_for(R.d, 256), 256, 0, st, R.ph_len.p, perm.p, R.d, lens_sorted.p);
        exclusive_scan<u32, u64>(lens_sorted.p, offs.p, R.d, offs.p + R.d, st);
        DevBuf<u64> first((u64)G + 1, st);
        GRL_LAUNCH("mg_bounds", 0, (mg2_bounds_kernel<u64>), 1, 32, 0, st, kp, R.d, (u32)G, first.p);
        std::vector<u64> hf((size_t)G + 1), ho((size_t)G + 1);
        d2h_mapped(hf.data(), first.p, ((size_t)G + 1) * 8, st);
        for (int g = 0; g <= G; g++) ho[(size_t)g] = d2h_scalar(offs.p + hf[(size_t)g], st);
        for (int g = 0; g < G; g++) { s_phr[(size_t)g] = hf[(size_t)g + 1] - hf[(size_t)g]; s_cel[(size_t)g] = ho[(size_t)g + 1] - ho[(size_t)g]; }
        s_cells.alloc(ho[(size_t)G] * sizeof(CellT) + 16, st);
        GRL_LAUNCH("pack_phrases", 0, (mg2_pack_kernel<CellT>), grid_for(R.d, 256), 256, 0, st, (const CellT*)c->text, R.ph_pos.p, R.ph_len.p, R.ph_freq.p, perm.p, offs.p, R.end_bits,
                   R.d, s_lens.p, s_counts.p, (CellT*)s_cells.p);
        GRL_CUDA(cudaStreamSynchronize(st));
    }
    clk.lap("pack by owner");
    // sizes: what every peer sends me, and the global parse length (termination: every string is one cell)
    std::vector<u64> r_phr((size_t)G), r_cel((size_t)G);
    bool done_global = false;
    u64 parse_total = 0, n_in_total = 0;
    {
        std::vector<u64> mine(2 * (size_t)G + 2);
        for (int g = 0; g < G; g++) { mine[(size_t)g] = s_phr[(size_t)g]; mine[(size_t)G + (size_t)g] = s_cel[(size_t)g]; }
        mine[2 * (size_t)G] = R.p;
        mine[2 * (size_t)G + 1] = R.n;
        const std::vector<u64> all = mg2_gather(cm, mine, st);
        for (int p = 0; p < G; p++) {
            const u64* row = all.data() + (size_t)p * (2 * (size_t)G + 2);
            r_phr[(size_t)p] = row[me];
            r_cel[(size_t)p] = row[G + me];
            parse_total += row[2 * G];
            n_in_total += row[2 * G + 1];
        }
        done_global = parse_total == c->mg_n_strings;
    }
    // ---- E1: phrases to their owners ----
    const u64 m = mg2_sum(r_phr), ncr = mg2_sum(r_cel);
    if (m >= 0xfffffff0ull) throw Error(GRLGPU_ERR_LIMIT, "more than 2^32 phrases arrived at one owner");
    DevBuf<u32> r_lens(m, st);
    DevBuf<u64> r_counts(m, st);
    DevBuf<u8> r_cells(ncr * sizeof(CellT) + 16, st);
    mg2_a2a_soa(cm, {{s_lens.p, r_lens.p, 4}, {s_counts.p, r_counts.p, 8}}, s_phr, r_phr, st);
    mg2_a2a<CellT>(cm, (const CellT*)s_cells.p, s_cel, (CellT*)r_cells.p, r_cel, st);
    GRL_CUDA(cudaStreamSynchronize(st));
    s_lens.release(); s_counts.release(); s_cells.release();
    clk.lap("E1 phrases to owners");
    // ---- M: owner-side dedup: my partition of the round's dictionary ----
    Mg2Part P(c);
    Round& PR = P.PR;
    DevBuf<u32> recv_dense(m, st);
    {
        DevBuf<u8> r_fin(m, st);
        GRL_LAUNCH("mg_strip_fin", m * 9, mg2_strip_fin_kernel, grid_for(m, 256), 256, 0, st, r_lens.p, m, r_fin.p);
        DevBuf<u64> r_offs(m + 1, st);
        exclusive_scan<u32, u64>(r_lens.p, r_offs.p, m, r_offs.p + m, st);
        {
            DevBuf<u64> len64(m, st), mx(1, st);
            mx.zero();
            GRL_LAUNCH("u32_to_u64", 0, u32_to_u64_kernel, grid_for(m, 256), 256, 0, st, r_lens.p, m, len64.p);
            GRL_LAUNCH("reduce_max_u64", 0, reduce_max_u64_kernel, 296, 256, 0, st, len64.p, m, mx.p);
            if (d2h_scalar(mx.p, st) >= HT_LEN_SAT) throw Error(GRLGPU_ERR_LIMIT, "multi-GPU rounds support phrases shorter than 2^24-1 cells");
            if (d2h_scalar(r_offs.p + m, st) != ncr) throw Error(GRLGPU_ERR_STATE, "received cell count does not match the received lengths");
        }
        const u64 cap = std::max<u64>(1024, (m + m / 2 + m / 10 + 255) / 256 * 256);
        if (cap > (1ull << 31) - 256) throw Error(GRLGPU_ERR_LIMIT, "phrase table would exceed 2^31 slots");
        DevBuf<ulonglong2> ptable(cap, st);
        GRL_LAUNCH("table_init", cap * 16, table_init_kernel, grid_for(cap, 256), 256, 0, st, ptable.p, cap);
        DevBuf<u32> overflow(1, st), recv_slot(m, st);
        overflow.zero();
        GRL_LAUNCH("pack_insert", 0, (pack_insert_kernel<CellT>), grid_for(m, 256), 256, 0, st, (const CellT*)r_cells.p, r_offs.p, r_lens.p, r_counts.p, m, ptable.p, cap, overflow.p,
                   recv_slot.p);
        if (d2h_scalar(overflow.p, st)) throw Error(GRLGPU_ERR_STATE, "partition table overflow");
        DevBuf<u32> occ_bits(cap / 32, st), pslots;
        GRL_LAUNCH("table_occupancy", cap * 16, table_occupancy_kernel, (unsigned)(cap / 256), 256, 0, st, ptable.p, cap, occ_bits.p);
        BitmapCompactor oc;
        PR.d = oc.count(occ_bits.p, cap, st);
        pslots.alloc(PR.d, st);
        if (PR.d) oc.write<u32>(nullptr, pslots.p);
        PR.ph_pos.alloc(PR.d, st);
        PR.ph_len.alloc(PR.d, st);
        PR.ph_freq.alloc(PR.d, st);
        GRL_LAUNCH("dict_meta", 0, dict_meta_kernel, grid_for(PR.d, 256), 256, 0, st, ptable.p, pslots.p, PR.d, (const u32*)nullptr, (const u32*)nullptr, (u64)0, PR.ph_pos.p,
                   PR.ph_len.p, PR.ph_freq.p);
        // the frequencies have been read: the count field now holds the slot's dense index, which every received phrase inherits
        GRL_LAUNCH("slot_dense", 0, slot_dense_kernel, grid_for(PR.d, 256), 256, 0, st, pslots.p, PR.d, ptable.p);
        GRL_LAUNCH("recv_dense", 0, recv_dense_kernel, grid_for(m, 256), 256, 0, st, recv_slot.p, m, ptable.p, recv_dense.p);
        P.p_fin.alloc(PR.d, st);
        GRL_LAUNCH("mg_part_fin", m * 6, mg2_part_fin_kernel, grid_for(m, 256), 256, 0, st, recv_dense.p, r_fin.p, m, P.p_fin.p);
        GRL_CUDA(cudaStreamSynchronize(st));
    }
    r_lens.release(); r_counts.release();
    PR.dict_text = r_cells.p;
    dict_offsets(PR);
    u64 d_g = 0, nE_g = 0, maxf_g = 0;
    {
        const std::vector<u64> all = mg2_gather(cm, std::vector<u64>{PR.d, PR.nE, PR.max_freq, PR.max_len}, st);
        for (int p = 0; p < G; p++) {
            d_g += all[(size_t)p * 4];
            nE_g += all[(size_t)p * 4 + 1];
            maxf_g = std::max(maxf_g, all[(size_t)p * 4 + 2]);
            P.max_freq_g = maxf_g;
            P.max_len_g = std::max(P.max_len_g, all[(size_t)p * 4 + 3]);
        }
    }
    clk.lap("M owner dedup");
    // ---- D .. E4: entries of my phrases, ranking by key range, rules by rank range ----
    const u64 A = c->alphabet;
    check_level_range(A, nE_g);  // every rank has the same A and nE_g: all of them refuse together
    P.sym_bits = bit_width64(A + 1);
    P.K = std::max(1, 64 / P.sym_bits);
    P.spare = P.sym_bits * P.K < 64 ? 64 - P.sym_bits * P.K : 0;
    if (level_is_wide(A, nE_g)) { mg2_gather<CellT, FIRST, u64>(c, P); clk.lap("D entries"); mg2_rank<u64>(c, cm, P, S); }
    else { mg2_gather<CellT, FIRST, u32>(c, P); clk.lap("D entries"); mg2_rank<u32>(c, cm, P, S); }
    clk.lap("(rank stages)");
    // ---- E5: metasymbols back to the ranks that saw the phrases, then the local rewrite ----
    {
        DevBuf<u64> reply(m, st), local_meta(R.d, st);
        if (m) GRL_LAUNCH("reply_meta", m * 20, reply_meta_kernel, grid_for(m, 256), 256, 0, st, recv_dense.p, m, (u64)0, (const u64*)P.p_meta.p, reply.p);
        mg2_a2a<u64>(cm, reply.p, r_phr, local_meta.p, s_phr, st);
        GRL_LAUNCH("apply_reply", R.d * 24, apply_reply_kernel, grid_for(R.d, 256), 256, 0, st, perm.p, R.occ_slots.p, local_meta.p, R.d, R.table.p);
        GRL_CUDA(cudaStreamSynchronize(st));
    }
    t_dict.stop();
    clk.lap("E5 metasymbols back");
    const u64 d_part = PR.d, nE_part = PR.nE;
    RoundTimes tm;
    tm.text = t_text.ms();
    tm.dict = t_dict.ms();
    c->lvl = DevLevel();  // the level lives in the slices
    c->lvl.sym_bytes = S.lvl.sym_bytes;
    finish_round(c, R, S.tot_global, S.n_pre_global, d_g, nE_g, maxf_g, tm, &t_all, out);
    clk.lap("rewrite");
    out->done = done_global ? 1u : 0u;  // the phase ends when EVERY rank's strings are single cells
    c->done = done_global;
    out->n_strings = c->mg_n_strings;
    c->mg_parse_len_local = R.p;
    c->mg_n_in_local = R.n;
    out->n_in = n_in_total;          // the scalars of `out` describe the global round; the local sizes are in grlgpu_slice_t
    out->parse_len = parse_total;
    // this rank's share of B_r (SURVEY.md 8d): its text in, its parse out, its partition of the dictionary
    out->algorithmic_bytes = R.n * (u64)out->cell_bytes_in + R.p * (u64)out->cell_bytes_out + nE_part * (u64)out->cell_bytes_in + 8 * d_part;
    c->lvl_n_in = ~0ull;
    c->is_suffix.release();
    c->mg_exchange_bytes = cm.bytes_sent - sent0;
}
