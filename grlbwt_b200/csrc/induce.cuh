// Induction phase ON THE DEVICE (SURVEY.md 8(f)-2, VERDICT r01 item 7): BWT_i from BWT_{i+1}, the level's grammar rules /
// hocc marks and its preliminary BWT, level by level from the deepest parse back to level 0 -- the semantics of the
// reference's infer_lvl_bwt (lib/exact_algo/exact_ind_phase.cpp:111-386; SURVEY.md App. B), reformulated as sorts, scans
// and sorted searches so that nothing is sequential:
//   A  chain expansion  every run (P, f) of BWT_{i+1} follows its grammar chain and emits (bucket g, left symbol l, f) tuples
//                       (+ (P, FROM_BWT, f) when P has a hocc bucket); the run keeps the chain's terminal symbol  (:143-258)
//   B  hocc buffer      = the tuples in bucket order, input order inside a bucket: one stable LSD radix sort on g
//                       (replaces compute_hocc_size :42-109 + the in-place bucket fills)
//   C  items            the output is the preliminary BWT with every hocc run replaced by its tuples: solved runs and literal
//                       tuples are literal items, "from BWT_{i+1}" runs and FROM_BWT tuples are slices of the rewritten
//                       BWT_{i+1} stream, consumed in order (:287-361). Item positions come from cross-ranking the two sorted
//                       lists (sorted binary searches), stream / output offsets from scans.
//   D  pieces           a stream slice expands into the stream runs it overlaps: the piece boundaries are the union of the
//                       item starts and the stream-run starts mapped into output coordinates (cross-ranking again)
//   E  maximal runs     adjacent pieces with equal symbols merge: head flags + compaction (:337-342,:352-357)
// All lengths and offsets are 32-bit: the device induction serves collections of fewer than 2^32 symbols whose levels use
// 32-bit symbols; anything else is induced by the host code (host/ind_phase_mt.hpp), which stays the general path.
// Included by grlgpu.cu inside its anonymous namespace.
#pragma once

constexpr u32 IND_STREAM = 0xffffffffu;  // item / tuple symbol: "take from the rewritten BWT_{i+1} stream"

// number of elements of the sorted array a[0, n) that are < x / <= x
__device__ __forceinline__ u32 ind_lower_bound(const u32* __restrict__ a, u32 n, u32 x) {
    u32 lo = 0, hi = n;
    while (lo < hi) { const u32 mid = (lo + hi) >> 1; if (a[mid] < x) lo = mid + 1; else hi = mid; }
    return lo;
}
__device__ __forceinline__ u32 ind_upper_bound(const u32* __restrict__ a, u32 n, u32 x) {
    u32 lo = 0, hi = n;
    while (lo < hi) { const u32 mid = (lo + hi) >> 1; if (a[mid] <= x) lo = mid + 1; else hi = mid; }
    return lo;
}

// deepest level: BWT_R = final parse (cells >> 1) in string order (parse2bwt_int, exact_ind_phase.cpp:621-635)
template <class CellT>
__global__ void __launch_bounds__(256) ind_parse_syms_kernel(const CellT* __restrict__ parse, u32 n, u32* __restrict__ sym) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sym[i] = (u32)((u64)parse[i] >> 1);
}
static __global__ void __launch_bounds__(256) ind_head_flags_kernel(const u32* __restrict__ sym, u32 n, u32* __restrict__ flags) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flags[i] = (i == 0 || sym[i] != sym[i - 1]) ? 1u : 0u;
}
// heads -> (symbol, start offset) of every maximal run; start[] gets one extra entry = total
static __global__ void __launch_bounds__(256) ind_compact_runs_kernel(const u32* __restrict__ sym, const u32* __restrict__ off, const u32* __restrict__ flags,
                                                                     const u32* __restrict__ excl, u32 n, u32 total, u32 n_runs, u32* __restrict__ run_sym,
                                                                     u32* __restrict__ run_start) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && flags[i]) { run_sym[excl[i]] = sym[i]; run_start[excl[i]] = off ? off[i] : i; }
    if (i == 0) run_start[n_runs] = total;
}
static __global__ void __launch_bounds__(256) ind_diff_kernel(const u32* __restrict__ start, u32 n, u32* __restrict__ len) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) len[i] = start[i + 1] - start[i];
}

// A: tuples per run, then the tuples themselves (exact_ind_phase.cpp:143-258)
static __global__ void __launch_bounds__(256) ind_chain_count_kernel(const u32* __restrict__ bsym, u32 m, const u32* __restrict__ rule_r, const u8* __restrict__ has_hocc,
                                                                    u32 alph3, u32* __restrict__ cnt) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const u32 P = bsym[i];
    u32 c = has_hocc[P] ? 1u : 0u;
    u32 r = rule_r[P];
    while (r >= alph3) { c++; r = rule_r[r - alph3]; }
    cnt[i] = c;
}
static __global__ void __launch_bounds__(256) ind_chain_emit_kernel(const u32* __restrict__ bsym, const u32* __restrict__ blen, u32 m, const u32* __restrict__ rule_l,
                                                                   const u32* __restrict__ rule_r, const u8* __restrict__ has_hocc, u32 alph3,
                                                                   const u64* __restrict__ toff, u32* __restrict__ tg, u32* __restrict__ tl, u32* __restrict__ tf,
                                                                   u32* __restrict__ tidx, u32* __restrict__ bsym2) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const u32 P = bsym[i], f = blen[i];
    u32 o = (u32)toff[i];
    if (has_hocc[P]) { tg[o] = P; tl[o] = IND_STREAM; tf[o] = f; tidx[o] = o; o++; }
    u32 l = rule_l[P], r = rule_r[P];
    while (r >= alph3) {
        const u32 g = r - alph3;
        tg[o] = g; tl[o] = l; tf[o] = f; tidx[o] = o; o++;
        l = rule_l[g];
        r = rule_r[g];
    }
    bsym2[i] = r;  // the chain's terminal symbol replaces the run's symbol
}
static __global__ void __launch_bounds__(256) ind_tuple_gather_kernel(const u32* __restrict__ perm, const u32* __restrict__ tl, const u32* __restrict__ tf, u32 n,
                                                                     u32* __restrict__ sl, u32* __restrict__ sf) {
    const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) { const u32 j = perm[k]; sl[k] = tl[j]; sf[k] = tf[j]; }
}
// C: preliminary-BWT runs: hocc flag, non-hocc flag, hocc length
template <class LenT>
__global__ void __launch_bounds__(256) ind_pre_flags_kernel(const u32* __restrict__ pre_sym, const LenT* __restrict__ pre_len, u32 n_pre, u32 hocc_dummy,
                                                            u32* __restrict__ nonh, u32* __restrict__ hlen, u32* __restrict__ len32) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pre) return;
    const bool h = pre_sym[i] == hocc_dummy;
    const u32 l = (u32)pre_len[i];
    nonh[i] = h ? 0u : 1u;
    hlen[i] = h ? l : 0u;
    len32[i] = l;
}
// non-hocc preliminary runs become items; position = non-hocc runs before + tuples before (those with hocc offset < pre_h)
static __global__ void __launch_bounds__(256) ind_items_from_pre_kernel(const u32* __restrict__ pre_sym, const u32* __restrict__ len32, const u32* __restrict__ nonh,
                                                                       const u32* __restrict__ nh_before, const u32* __restrict__ pre_h, u32 n_pre,
                                                                       const u32* __restrict__ cum_h, u32 n_t, u32 bwt_dummy, u32* __restrict__ it_sym,
                                                                       u32* __restrict__ it_len, u32* err) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pre) return;
    const u32 before = ind_lower_bound(cum_h, n_t, pre_h[i]);
    // every preliminary run must start on a tuple boundary of the hocc buffer (a hocc run covers whole buckets)
    if (before < n_t ? cum_h[before] != pre_h[i] : pre_h[i] != cum_h[n_t]) atomicExch(err, 1u);
    if (!nonh[i]) return;
    const u32 pos = nh_before[i] + before;
    it_sym[pos] = pre_sym[i] == bwt_dummy ? IND_STREAM : pre_sym[i];
    it_len[pos] = len32[i];
}
// tuples become items; position = tuple index + non-hocc runs before the hocc run that owns the tuple
static __global__ void __launch_bounds__(256) ind_items_from_tuples_kernel(const u32* __restrict__ sl, const u32* __restrict__ sf, const u32* __restrict__ cum_h, u32 n_t,
                                                                          const u32* __restrict__ pre_h, const u32* __restrict__ nh_before, u32 n_pre,
                                                                          u32* __restrict__ it_sym, u32* __restrict__ it_len) {
    const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_t) return;
    // owner = last preliminary run whose hocc offset is <= the tuple's (runs that are not hocc repeat their successor's offset and
    // sit BEFORE it, so the last one with pre_h <= x is the hocc run holding x)
    const u32 owner = ind_upper_bound(pre_h, n_pre, cum_h[k]) - 1;
    const u32 pos = k + nh_before[owner];
    it_sym[pos] = sl[k];
    it_len[pos] = sf[k];
}
static __global__ void __launch_bounds__(256) ind_item_stream_len_kernel(const u32* __restrict__ it_sym, const u32* __restrict__ it_len, u32 n, u32* __restrict__ slen) {
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) slen[t] = it_sym[t] == IND_STREAM ? it_len[t] : 0u;
}
// D: stream-run starts: containing item, coincidence with an item start
static __global__ void __launch_bounds__(256) ind_run_item_kernel(const u32* __restrict__ cum_s, u32 m, const u32* __restrict__ it_s, u32 n_items, u32* __restrict__ citem,
                                                                 u32* __restrict__ ncflag, u32* rcnt) {
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const u32 x = cum_s[j];
    const u32 c = ind_upper_bound(it_s, n_items, x) - 1;  // last item whose stream offset is <= x: the stream item that holds x
    citem[j] = c;
    ncflag[j] = it_s[c] == x ? 0u : 1u;
    // runs held by item c: their exclusive prefix over the items is, for every item t, the number of stream runs that start before
    // t's stream offset (a run starts before it_s[t] exactly when its item comes before t) -- no search from the items' side
    atomicAdd(&rcnt[c], 1u);
}
static __global__ void __launch_bounds__(256) ind_pieces_from_runs_kernel(const u32* __restrict__ cum_s, const u32* __restrict__ bsym2, u32 m, const u32* __restrict__ citem,
                                                                         const u32* __restrict__ ncflag, const u32* __restrict__ nc_before,
                                                                         const u32* __restrict__ it_s, const u32* __restrict__ it_o, u32* __restrict__ p_sym,
                                                                         u32* __restrict__ p_off) {
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m || !ncflag[j]) return;
    const u32 c = citem[j], q = c + 1 + nc_before[j];
    p_sym[q] = bsym2[j];
    p_off[q] = it_o[c] + (cum_s[j] - it_s[c]);
}
static __global__ void __launch_bounds__(256) ind_pieces_from_items_kernel(const u32* __restrict__ it_sym, const u32* __restrict__ it_s, const u32* __restrict__ it_o,
                                                                          u32 n_items, const u32* __restrict__ cum_s, const u32* __restrict__ bsym2, u32 m,
                                                                          const u32* __restrict__ runs_before, const u32* __restrict__ nc_before,
                                                                          u32* __restrict__ p_sym, u32* __restrict__ p_off) {
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_items) return;
    const u32 r = runs_before[t];                        // stream runs that start before the item's stream offset
    const u32 q = t + nc_before[r];
    u32 sym = it_sym[t];
    if (sym == IND_STREAM) sym = bsym2[(r < m && cum_s[r] == it_s[t]) ? r : r - 1];  // the stream run that holds the slice's first symbol
    p_sym[q] = sym;
    p_off[q] = it_o[t];
}

// LSD radix sort of (u32 key, u32 value) pairs on key bits [0, n_bits)

// the run-length BWT as .rl_bwt records (rl_bwt_io.hpp; the reference's bwt_buff_writer, external/cdt/include/bwt_io.h): sb symbol
// bytes + fb length bytes per run, little endian. A CTA packs IND_PACK_RUNS runs into shared memory and stores them as 16-byte
// vectors (IND_PACK_RUNS * rec is a multiple of 16, so every CTA starts on a 16-byte boundary of the record stream).
constexpr int IND_PACK_RUNS = 1024;
static __global__ void __launch_bounds__(256) ind_pack_records_kernel(const u32* __restrict__ sym, const u32* __restrict__ len, u64 first, u64 n, int sb, int fb,
                                                                      unsigned char* __restrict__ out, u32* err) {
    extern __shared__ __align__(16) unsigned char pk_smem[];
    const int rec = sb + fb;
    const u64 r0 = (u64)blockIdx.x * IND_PACK_RUNS;
    const u32 here = (u32)((n - r0) < (u64)IND_PACK_RUNS ? (n - r0) : (u64)IND_PACK_RUNS);
    for (u32 k = threadIdx.x; k < here; k += 256) {
        const u64 s = sym[first + r0 + k], l = len[first + r0 + k];
        if ((sb < 8 && (s >> (8 * sb))) || (fb < 8 && (l >> (8 * fb)))) atomicExch(err, 1u);
        unsigned char* q = pk_smem + (size_t)k * rec;
        for (int b = 0; b < sb; b++) q[b] = (unsigned char)(s >> (8 * b));
        for (int b = 0; b < fb; b++) q[sb + b] = (unsigned char)(l >> (8 * b));
    }
    __syncthreads();
    const u32 bytes = here * (u32)rec, nvec = bytes >> 4;
    unsigned char* dst = out + r0 * (u64)rec;
    for (u32 v = threadIdx.x; v < nvec; v += 256) reinterpret_cast<uint4*>(dst)[v] = reinterpret_cast<const uint4*>(pk_smem)[v];
    for (u32 b = (nvec << 4) + threadIdx.x; b < bytes; b += 256) dst[b] = pk_smem[b];
}

inline u32 ind_scan_total(const u32* in, u32* out, u32 n, cudaStream_t st) {  // exclusive scan; out may have n + 1 entries (total stored at out[n])
    exclusive_scan<u32, u32>(in, out, n, out + n, st);
    return d2h_scalar(out + n, st);
}

// (symbols, run starts with a trailing total) of the maximal runs of a piece / symbol sequence
inline void ind_maximal_runs(const u32* sym, const u32* off, u32 n, u32 total, IndBwt& out, cudaStream_t st) {
    DevBuf<u32> flags(n, st), excl((u64)n + 1, st);
    GRL_LAUNCH("ind_head_flags", n * 8, ind_head_flags_kernel, grid_for(n, 256), 256, 0, st, sym, n, flags.p);
    const u32 n_runs = ind_scan_total(flags.p, excl.p, n, st);
    DevBuf<u32> start((u64)n_runs + 1, st);
    out.sym.alloc(n_runs, st);
    out.len.alloc(n_runs, st);
    GRL_LAUNCH("ind_compact_runs", n * 16, ind_compact_runs_kernel, grid_for(n, 256), 256, 0, st, sym, off, flags.p, excl.p, n, total, n_runs, out.sym.p, start.p);
    GRL_LAUNCH("ind_diff", n_runs * 8, ind_diff_kernel, grid_for(n_runs, 256), 256, 0, st, start.p, n_runs, out.len.p);
    out.n_runs = n_runs;
    out.n_syms = total;
    GRL_CUDA(cudaStreamSynchronize(st));
}

// one level step BWT_{i+1} -> BWT_i; throws GRLGPU_ERR_STATE when the level's artefacts disagree
inline void ind_level_step(IndBwt& bwt, const IndLevel& K, cudaStream_t st, bool trace) {
    const DevLevel& L = K.lvl;
    const u32 A = (u32)K.alphabet, alph3 = A + 3, bwt_dummy = A + 1, hocc_dummy = A + 2;
    const u32 m = bwt.n_runs, n_pre = (u32)L.n_pre;
    const u32* rule_l = (const u32*)L.rule_l.p;
    const u32* rule_r = (const u32*)L.rule_r.p;
    const u32* pre_sym = (const u32*)L.pre_sym.p;
    // ---- A: chain expansion ----
    DevBuf<u32> tcnt(m, st), bsym2(m, st);
    DevBuf<u64> toff((u64)m + 1, st);
    GRL_LAUNCH("ind_chain_count", m * 24, ind_chain_count_kernel, grid_for(m, 256), 256, 0, st, bwt.sym.p, m, rule_r, L.has_hocc.p, alph3, tcnt.p);
    exclusive_scan<u32, u64>(tcnt.p, toff.p, m, toff.p + m, st);
    const u64 n_t64 = d2h_scalar(toff.p + m, st);
    if (n_t64 >= 0xfffffff0ull) throw Error(GRLGPU_ERR_LIMIT, "induction on the device: more than 2^32 hocc tuples in one level");
    tcnt.release();
    const u32 n_t = (u32)n_t64;
    DevBuf<u32> sl(n_t, st), sf(n_t, st);
    {
        DevBuf<u32> tg(n_t, st), tl(n_t, st), tf(n_t, st), tidx(n_t, st), tg_alt(n_t, st), tidx_alt(n_t, st);
        GRL_LAUNCH("ind_chain_emit", m * 24 + n_t * 16, ind_chain_emit_kernel, grid_for(m, 256), 256, 0, st, bwt.sym.p, bwt.len.p, m, rule_l, rule_r, L.has_hocc.p, alph3, toff.p, tg.p,
                   tl.p, tf.p, tidx.p, bsym2.p);
        // ---- B: hocc buffer = tuples in bucket order, input order inside a bucket ----
        u32 *kp = tg.p, *vp = tidx.p, *ka = tg_alt.p, *va = tidx_alt.p;
        radix_sort_pairs_u32(&kp, &vp, &ka, &va, n_t, std::max(1, bit_width64(L.tot ? L.tot - 1 : 0)), st);
        GRL_LAUNCH("ind_tuple_gather", n_t * 20, ind_tuple_gather_kernel, grid_for(n_t, 256), 256, 0, st, vp, tl.p, tf.p, n_t, sl.p, sf.p);
        GRL_CUDA(cudaStreamSynchronize(st));
    }
    toff.release();
    // ---- C: items ----
    DevBuf<u32> cum_h((u64)n_t + 1, st);
    const u32 hocc_total = ind_scan_total(sf.p, cum_h.p, n_t, st);
    DevBuf<u32> nonh(n_pre, st), hlen(n_pre, st), len32(n_pre, st), nh_before((u64)n_pre + 1, st), pre_h((u64)n_pre + 1, st);
    GRL_LAUNCH("ind_pre_flags", n_pre * 24, (ind_pre_flags_kernel<u64>), grid_for(n_pre, 256), 256, 0, st, pre_sym, L.pre_len.p, n_pre, hocc_dummy, nonh.p, hlen.p, len32.p);
    const u32 n_nonh = ind_scan_total(nonh.p, nh_before.p, n_pre, st);
    const u32 hocc_pre = ind_scan_total(hlen.p, pre_h.p, n_pre, st);
    if (hocc_pre != hocc_total) throw Error(GRLGPU_ERR_STATE, "induction: hocc buffer and preliminary BWT disagree");
    const u32 n_items = n_nonh + n_t;
    DevBuf<u32> it_sym(n_items, st), it_len(n_items, st), err(1, st);
    err.zero();
    GRL_LAUNCH("ind_items_pre", n_pre * 40, ind_items_from_pre_kernel, grid_for(n_pre, 256), 256, 0, st, pre_sym, len32.p, nonh.p, nh_before.p, pre_h.p, n_pre, cum_h.p, n_t, bwt_dummy,
               it_sym.p, it_len.p, err.p);
    GRL_LAUNCH("ind_items_tuples", n_t * 40, ind_items_from_tuples_kernel, grid_for(n_t, 256), 256, 0, st, sl.p, sf.p, cum_h.p, n_t, pre_h.p, nh_before.p, n_pre, it_sym.p, it_len.p);
    if (d2h_scalar(err.p, st)) throw Error(GRLGPU_ERR_STATE, "induction: a preliminary run starts inside a hocc tuple");
    sl.release(); sf.release(); cum_h.release(); nonh.release(); hlen.release(); len32.release(); nh_before.release(); pre_h.release();
    DevBuf<u32> it_s((u64)n_items + 1, st), it_o((u64)n_items + 1, st);
    {
        DevBuf<u32> slen(n_items, st);
        GRL_LAUNCH("ind_item_stream_len", n_items * 12, ind_item_stream_len_kernel, grid_for(n_items, 256), 256, 0, st, it_sym.p, it_len.p, n_items, slen.p);
        const u32 stream_total = ind_scan_total(slen.p, it_s.p, n_items, st);
        if (stream_total != bwt.n_syms) throw Error(GRLGPU_ERR_STATE, "induction: stream and preliminary BWT disagree");
    }
    const u32 n_out = ind_scan_total(it_len.p, it_o.p, n_items, st);
    it_len.release();
    // ---- D: pieces ----
    DevBuf<u32> cum_s((u64)m + 1, st), citem(m, st), ncflag(m, st), nc_before((u64)m + 1, st), runs_before((u64)n_items + 1, st);
    ind_scan_total(bwt.len.p, cum_s.p, m, st);
    runs_before.zero();
    GRL_LAUNCH("ind_run_item", m * 40, ind_run_item_kernel, grid_for(m, 256), 256, 0, st, cum_s.p, m, it_s.p, n_items, citem.p, ncflag.p, runs_before.p);
    ind_scan_total(runs_before.p, runs_before.p, n_items, st);
    const u32 n_nc = ind_scan_total(ncflag.p, nc_before.p, m, st);
    const u32 n_pieces = n_items + n_nc;
    DevBuf<u32> p_sym(n_pieces, st), p_off(n_pieces, st);
    GRL_LAUNCH("ind_pieces_runs", m * 40, ind_pieces_from_runs_kernel, grid_for(m, 256), 256, 0, st, cum_s.p, bsym2.p, m, citem.p, ncflag.p, nc_before.p, it_s.p, it_o.p, p_sym.p, p_off.p);
    GRL_LAUNCH("ind_pieces_items", n_items * 40, ind_pieces_from_items_kernel, grid_for(n_items, 256), 256, 0, st, it_sym.p, it_s.p, it_o.p, n_items, cum_s.p, bsym2.p, m,
               runs_before.p, nc_before.p, p_sym.p, p_off.p);
    GRL_CUDA(cudaStreamSynchronize(st));
    it_sym.release(); it_s.release(); it_o.release(); cum_s.release(); citem.release(); ncflag.release(); nc_before.release(); bsym2.release(); runs_before.release();
    // ---- E: maximal runs ----
    IndBwt next;
    ind_maximal_runs(p_sym.p, p_off.p, n_pieces, n_out, next, st);
    if (trace) fprintf(stderr, "[grlgpu] induction: level alphabet %u: %u runs -> %u tuples, %u items, %u pieces -> %u runs of %u symbols\n", A, m, n_t, n_items, n_pieces, next.n_runs, n_out);
    bwt = std::move(next);
}
