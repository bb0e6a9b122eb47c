// Search of a BCR BWT ON THE DEVICE: a .rl_bwt image kept as a run-length FM-index, queried for count and locate.
//   load     the LF table of invert.cuh (part a, shared), kept with its run arrays and the symbol-sorted run order; a symbol
//            directory (per distinct symbol: its slice of that order and C[c]) from head flags over the sorted symbols; psi = LF^-1
//   count    backward search, one thread per pattern, from its last symbol; LF_c(i) = C[c] + rank_c(BWT, i) for i in [0, n]:
//            the run k holding i (upper bound on the run starts, k = r for i = n) gives F[k] + i - start[k] when its symbol is c,
//            otherwise the last run q < k of c's slice (binary search) gives F[q] + len[q], or C[c] when there is none
//   locate   one thread per occurrence (row j of some [sp, ep)), offsets of the occurrences = exclusive scan of ep - sp in u64:
//            the offset p = LF steps from j to a row whose BWT symbol is the separator; the string k = the first row < N that
//            psi steps reach from j (row k < N is $_k, the end of string k); both walks bounded by B (inv_walk_bound). A longer
//            walk switches the call to a table of (k, p) for every row, built once per index by pointer jumping (invert.cuh,
//            part c: p = d, k = the string whose chain from row k ends at succ) and kept for every later call.
//   extract  one thread per request (k, from, len), S_k[from .. e) with e = min(from + len, L_k): the walk counts L_k by LF steps
//            from row k (the count pass of invert.cuh with the request's k, bound B), then walks again from row k at position
//            L_k, writing the cells below e backwards through InvStage. A string longer than B switches the call to samples: the
//            row at every FM_EXTRACT_SAMPLE-th position of every string, taken from the locate table (built here when no locate
//            built it) and kept for every later call; the walk then starts at the first sample at or after e.
//   approx   count / locate with at most k <= 3 substitutions: one thread per pattern, a depth-first backward search over at most
//            k + 1 frames (fm_approx_kernel), hits appended to a pool, sorted by (pattern, sp); locate runs on the hits' intervals
//   lcp      LCP array of every row: SA and the text T from the walk per string (or the locate table), then one warp per
//            irreducible row (a run head or a separator symbol) compares T at SA[j] and SA[j - 1]; the other rows follow from
//            PLCP[i] + i = PLCP[i - 1] + (i - 1), filled in by a max-scan over text positions, and are gathered back to rows
// Convention of reverse_bwt and grlgpu_invert: the separator is the smallest symbol of a non-empty record, N its count, strings in
// input order. A pattern containing the separator or a symbol outside the directory has no occurrence; every empty interval is
// reported as sp = ep = 0 (the host tool fm_query does the same). Positions and symbols are 32-bit, as for the inversion.
// Included by grlgpu.cu inside its anonymous namespace, after invert.cuh.
#pragma once

constexpr u32 FM_OVER_POLL = 256;  // locate walk: steps between two reads of the "some walk is over the bound" flag
// extract: one sampled row per FM_EXTRACT_SAMPLE positions of a string (n / 16 bytes, plus 4 bytes per string), so a request walks at
// most FM_EXTRACT_SAMPLE - 1 steps more than it writes (DESIGN.md §12, "Extract")
constexpr u32 FM_EXTRACT_SAMPLE = 64;

struct FmView {  // device arrays of a loaded index, passed to the search kernels by value
    const u32 *start, *sym, *len, *F, *order, *dir_sym, *dir_first, *dir_C;
    u32 n, n_runs, n_dir, sep;
};

// position of symbol v in the directory, or n_dir when the index has no record of it (or v is the separator)
__device__ __forceinline__ u32 fm_dir_find(const FmView& x, u64 v) {
    if ((v >> 32) || (u32)v == x.sep) return x.n_dir;
    const u32 d = ind_lower_bound(x.dir_sym, x.n_dir, (u32)v);
    return (d < x.n_dir && x.dir_sym[d] == (u32)v) ? d : x.n_dir;
}
// LF_c(i) = C[c] + rank_c(BWT, i), i in [0, n], c = dir_sym[d]
__device__ __forceinline__ u32 fm_lf_c(const FmView& x, u32 d, u32 i) {
    const u32 c = x.dir_sym[d];
    const u32 k = ind_upper_bound(x.start, x.n_runs + 1, i) - 1;  // start[n_runs] = n: k = n_runs for i = n
    if (k < x.n_runs && x.sym[k] == c) return x.F[k] + (i - x.start[k]);
    const u32 lo = x.dir_first[d], m = ind_lower_bound(x.order + lo, x.dir_first[d + 1] - lo, k);  // runs of c before run k
    if (m == 0) return x.dir_C[d];
    const u32 q = x.order[lo + m - 1];
    return x.F[q] + x.len[q];
}

// one thread per pattern: sp_ep[2q], sp_ep[2q + 1]
template <class CellT>
__global__ void __launch_bounds__(INV_THREADS) fm_count_kernel(FmView x, const CellT* __restrict__ pat, const u64* __restrict__ pat_off, u64 n_pat, u64* __restrict__ sp_ep) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_pat) return;
    u32 sp = 0, ep = x.n;
    for (u64 a = pat_off[q + 1]; a > pat_off[q];) {  // the pattern's cells, last first
        const u32 d = fm_dir_find(x, (u64)pat[--a]);
        if (d == x.n_dir) { sp = ep = 0; break; }
        sp = fm_lf_c(x, d, sp);
        ep = fm_lf_c(x, d, ep);
        if (sp >= ep) { sp = ep = 0; break; }
    }
    sp_ep[2 * q] = sp;
    sp_ep[2 * q + 1] = ep;
}
// approximate search (DESIGN.md §12, "Approximate search"): one thread per pattern, depth-first over the substitutions, hits
// appended to a pool of `cap` entries through counters[0] (which keeps counting past cap). Frame j holds the state after j
// substitutions: t cells of the pattern are still to match (cells 0 .. t - 1), [sp, ep) is the interval of the suffix matched so
// far, [ra, rb) the runs holding it, cur the next substitution to try at cell t - 1 (a run of [ra, rb) when they are fewer than
// the directory's symbols, else a directory index). Exact steps move a frame's own t down; a substitution pushes frame j + 1.
constexpr u32 FM_APPROX_MAX_K = 3;
struct FmFrame { u32 t, sp, ep, cur, ra, rb; };
__device__ __forceinline__ FmFrame fm_frame(const FmView& x, u32 t, u32 sp, u32 ep, bool subst) {
    if (!subst || t == 0) return FmFrame{t, sp, ep, 0, 0, 0};  // no substitution will be tried: the runs are not needed
    return FmFrame{t, sp, ep, 0, ind_upper_bound(x.start, x.n_runs + 1, sp) - 1, ind_upper_bound(x.start, x.n_runs + 1, ep - 1)};
}
template <class CellT>
__global__ void __launch_bounds__(INV_THREADS) fm_approx_kernel(FmView x, const CellT* __restrict__ pat, const u64* __restrict__ pat_off, u64 n_pat, u32 kmax,
                                                                u64 cap, u64* __restrict__ key, u32* __restrict__ slot, u64* __restrict__ ep_d, u64* __restrict__ cnt,
                                                                u64* counters /* [0] hits, [1] LF_c evaluations */) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_pat) return;
    const CellT* P = pat + pat_off[q];
    const u64 m = pat_off[q + 1] - pat_off[q];
    u64 hits = 0, lf = 0;
    FmFrame f[FM_APPROX_MAX_K + 1];
    int j = 0;
    if (m < x.n) f[0] = fm_frame(x, (u32)m, 0, x.n, kmax > 0);
    else j = -1;  // a window inside a string has fewer cells than the BWT has rows
    // Each pass either emits a hit and pops, tries one substitution (at most sigma per cell and frame), takes one exact step (at
    // most m per frame) or pops: at most kmax + 1 <= 4 frames live, so the loop ends after O(m * sigma) passes per frame pushed.
    while (j >= 0) {
        FmFrame& F = f[j];
        if (F.t == 0) {  // the whole pattern is matched with j substitutions
            const u64 s = atomicAdd((unsigned long long*)counters, 1ull);
            if (s < cap) { key[s] = (q << 32) | F.sp; slot[s] = (u32)s; ep_d[s] = ((u64)j << 32) | F.ep; }
            hits++;
            j--;
            continue;
        }
        const u64 own = (u64)P[F.t - 1];
        if ((u32)j < kmax) {  // substitutions at cell t - 1: symbols other than the separator and the cell's own
            bool found = false;
            u32 csp = 0, cep = 0;
            if (F.rb - F.ra < x.n_dir) {  // the symbols of the runs holding [sp, ep), each tried at its first run there
                while (!found && F.ra + F.cur < F.rb) {  // at most rb - ra < sigma candidates
                    const u32 r = F.ra + F.cur++, c = x.sym[r];
                    if (c == x.sep || (u64)c == own) continue;
                    const u32 first = x.F[r] + (max(F.sp, x.start[r]) - x.start[r]);  // LF_c(sp) when r is c's first run in [sp, ep)
                    if (F.rb - F.ra == 1) {  // one run: LF_c = F + the offset in the run, no search
                        csp = first;
                        cep = x.F[r] + (F.ep - x.start[r]);
                        lf += 2;
                        found = true;
                        continue;
                    }
                    const u32 d = fm_dir_find(x, c);
                    csp = fm_lf_c(x, d, F.sp);
                    lf++;
                    if (csp != first) continue;  // c has an earlier run in the interval, where it was tried
                    cep = fm_lf_c(x, d, F.ep);
                    lf++;
                    found = true;  // non-empty: run r holds c inside [sp, ep)
                }
            } else {
                for (; !found && F.cur < x.n_dir; F.cur++) {  // at most sigma candidates
                    const u32 c = x.dir_sym[F.cur];
                    if (c == x.sep || (u64)c == own) continue;
                    csp = fm_lf_c(x, F.cur, F.sp);
                    cep = fm_lf_c(x, F.cur, F.ep);
                    lf += 2;
                    found = csp < cep;
                }
            }
            if (found) {
                f[j + 1] = fm_frame(x, F.t - 1, csp, cep, (u32)j + 1 < kmax);
                j++;
                continue;
            }
        }
        // no substitution left at this cell: the exact step
        const u32 d = fm_dir_find(x, own);
        if (d == x.n_dir) { j--; continue; }
        const u32 sp = fm_lf_c(x, d, F.sp), ep = fm_lf_c(x, d, F.ep);
        lf += 2;
        if (sp >= ep) { j--; continue; }
        F = fm_frame(x, F.t - 1, sp, ep, (u32)j < kmax);
    }
    cnt[q] = hits;
    atomicAdd((unsigned long long*)counters + 1, (unsigned long long)lf);
}
// hits in (pattern, sp) order: slot s of the pool -> sp_ep[2i], sp_ep[2i + 1], mm[i]
static __global__ void __launch_bounds__(INV_THREADS) fm_approx_gather_kernel(const u64* __restrict__ key, const u32* __restrict__ slot, const u64* __restrict__ ep_d, u64 n_hits,
                                                                              u64* __restrict__ sp_ep, u8* __restrict__ mm) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_hits) return;
    const u64 e = ld_gather8(ep_d + slot[i]);
    sp_ep[2 * i] = (u32)key[i];
    sp_ep[2 * i + 1] = (u32)e;
    mm[i] = (u8)(e >> 32);
}
// approximate locate: occurrence o takes the d of its hit; pattern q's occurrences start where its first hit's do
static __global__ void __launch_bounds__(INV_THREADS) fm_approx_occ_mm_kernel(const u64* __restrict__ hit_occ, u64 n_hits, const u8* __restrict__ hit_mm, u64 n_occ,
                                                                              u8* __restrict__ occ_mm) {
    const u64 o = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n_occ) return;
    u64 lo = 0, hi = n_hits;  // last h with hit_occ[h] <= o
    while (hi - lo > 1) { const u64 mid = (lo + hi) >> 1; if (hit_occ[mid] <= o) lo = mid; else hi = mid; }
    occ_mm[o] = hit_mm[lo];
}
static __global__ void __launch_bounds__(INV_THREADS) fm_approx_occ_off_kernel(const u64* __restrict__ hit_occ, const u64* __restrict__ hit_off, u64 n_pat, u64* __restrict__ occ_off) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q <= n_pat) occ_off[q] = hit_occ[hit_off[q]];
}

static __global__ void __launch_bounds__(INV_THREADS) fm_occ_count_kernel(const u64* __restrict__ sp_ep, u64 n_pat, u64* __restrict__ cnt) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q < n_pat) cnt[q] = sp_ep[2 * q + 1] - sp_ep[2 * q];
}
// row of occurrence o: the pattern q with occ_off[q] <= o < occ_off[q + 1], then sp + the rank inside [sp, ep)
__device__ __forceinline__ u32 fm_occ_row(const u64* __restrict__ sp_ep, const u64* __restrict__ occ_off, u64 n_pat, u64 o) {
    u64 lo = 0, hi = n_pat;  // last q with occ_off[q] <= o (occ_off[0] = 0 <= o)
    while (hi - lo > 1) { const u64 mid = (lo + hi) >> 1; if (occ_off[mid] <= o) lo = mid; else hi = mid; }
    return (u32)(sp_ep[2 * lo] + (o - occ_off[lo]));
}
// walk: at most `bound` LF steps for p and `bound` psi steps for k; a longer walk sets *over and leaves the occurrence unwritten.
// Once *over is set the whole call goes to the table, so every thread stops: at its start, and every FM_OVER_POLL steps of a walk.
static __global__ void __launch_bounds__(INV_THREADS) fm_locate_walk_kernel(const u64* __restrict__ E, const u32* __restrict__ psi, u32 N, u32 sep, const u64* __restrict__ sp_ep,
                                                                            const u64* __restrict__ occ_off, u64 n_pat, u64 n_occ, u32 bound, u32* __restrict__ str_id,
                                                                            u32* __restrict__ str_pos, u32* over) {
    const u64 o = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n_occ) return;
    const volatile u32* over_v = over;
    if (*over_v) return;
    const u32 j = fm_occ_row(sp_ep, occ_off, n_pat, o);
    u32 r = j, p = 0;
    for (; p < bound; p++) {  // bounded by `bound`
        const u64 e = ld_gather8(E + r);
        if (inv_sym(e) == sep) break;
        r = inv_lf(e);
        if ((p & (FM_OVER_POLL - 1)) == FM_OVER_POLL - 1 && *over_v) return;
    }
    u32 k = j, f = 0;
    for (; f < bound; f++) {  // bounded by `bound`
        k = ld_gather4(psi + k);
        if (k < N) break;
        if ((f & (FM_OVER_POLL - 1)) == FM_OVER_POLL - 1 && *over_v) return;
    }
    if (p == bound || f == bound) { atomicExch(over, 1u); return; }
    str_id[o] = k;
    str_pos[o] = p;
}
static __global__ void __launch_bounds__(INV_THREADS) fm_locate_table_kernel(const u64* __restrict__ doc, const u64* __restrict__ sp_ep, const u64* __restrict__ occ_off, u64 n_pat,
                                                                             u64 n_occ, u32* __restrict__ str_id, u32* __restrict__ str_pos) {
    const u64 o = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n_occ) return;
    const u64 t = ld_gather8(doc + fm_occ_row(sp_ep, occ_off, n_pat, o));
    str_id[o] = (u32)(t >> 32);
    str_pos[o] = (u32)t;
}

// load: C[c] of every directory entry = F row of the first run of its slice
static __global__ void __launch_bounds__(INV_THREADS) fm_dir_c_kernel(const u32* __restrict__ dir_first, const u32* __restrict__ order, const u32* __restrict__ F, u32 n_dir,
                                                                      u32* __restrict__ dir_C) {
    const u32 d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d < n_dir) dir_C[d] = F[order[dir_first[d]]];
}
static __global__ void __launch_bounds__(INV_THREADS) fm_psi_kernel(const u64* __restrict__ E, u32 n, u32* __restrict__ psi) {
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) psi[inv_lf(E[j])] = j;
}
// locate table from converged pointer jumping: doc[j] = {owner[succ] << 32 | d}; a chain that ends on a row that is not a
// separator row, or on one no string i < N reaches, lies on a cycle without separator (*bad)
static __global__ void __launch_bounds__(INV_THREADS) fm_doc_kernel(const u64* __restrict__ E, const u64* __restrict__ P, const u32* __restrict__ owner, u32 n, u32 N, u32 sep,
                                                                    u64* __restrict__ doc, u32* bad) {
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const u64 p = P[j];
    const u32 s = (u32)p, k = ld_gather4(owner + s);
    if (inv_sym(ld_gather8(E + s)) != sep || k >= N) { atomicExch(bad, 1u); return; }
    doc[j] = ((u64)k << 32) | (p >> 32);
}

// extract samples from the locate table: string k (row k < N has offset L_k) has L_k / S + 1 samples, at offsets 0, S, ..
static __global__ void __launch_bounds__(INV_THREADS) fm_samp_len_kernel(const u64* __restrict__ doc, u32 N, u32* __restrict__ cnt) {
    const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < N) cnt[k] = (u32)doc[k] / FM_EXTRACT_SAMPLE + 1;
}
static __global__ void __launch_bounds__(INV_THREADS) fm_samp_fill_kernel(const u64* __restrict__ doc, u32 n, const u32* __restrict__ samp_off, u32* __restrict__ samp) {
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const u64 t = doc[j];
    const u32 p = (u32)t;
    if (p % FM_EXTRACT_SAMPLE == 0) samp[ld_gather4(samp_off + (u32)(t >> 32)) + p / FM_EXTRACT_SAMPLE] = j;
}
// request q: L_k of its string (read from the locate table into Lq when doc is given, else left there by the count pass) and its
// cell count e - from, e = min(from + len, L_k) in 64 bits (0 when from >= e)
static __global__ void __launch_bounds__(INV_THREADS) fm_extract_size_kernel(const u32* __restrict__ str_id, const u32* __restrict__ from, const u32* __restrict__ len, u32 n_req,
                                                                             const u64* __restrict__ doc, u32* __restrict__ Lq, u64* __restrict__ cnt) {
    const u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_req) return;
    u32 L;
    if (doc) Lq[q] = L = (u32)ld_gather8(doc + str_id[q]);
    else L = Lq[q];
    const u64 e = min((u64)from[q] + len[q], (u64)L);
    cnt[q] = from[q] < e ? e - from[q] : 0;
}
// request q: walk LF back from a row at a known position of string k down to position from, writing the cells of the positions
// below e: from row k at L_k (the end of the string), or, with samples, from the first sampled position at or after e that lies
// inside the string. The row at position p has BWT = S_k[p - 1], so a step from p emits S_k[p - 1].
template <class CellT>
__global__ void __launch_bounds__(INV_THREADS) fm_extract_write_kernel(const u64* __restrict__ E, const u32* __restrict__ str_id, const u32* __restrict__ from,
                                                                       const u32* __restrict__ len, const u32* __restrict__ Lq, const u64* __restrict__ out_off, u32 n_req,
                                                                       const u32* __restrict__ samp, const u32* __restrict__ samp_off, u8* __restrict__ out) {
    const u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_req) return;
    const u32 k = str_id[q], L = Lq[q], f = from[q];
    const u32 e = (u32)min((u64)f + len[q], (u64)L);
    if (f >= e) return;
    u32 r = k, p = L;
    if (samp) {
        const u32 s = (u32)(((u64)e + FM_EXTRACT_SAMPLE - 1) / FM_EXTRACT_SAMPLE);
        if ((u64)s * FM_EXTRACT_SAMPLE < L) { r = ld_gather4(samp + ld_gather4(samp_off + k) + s); p = s * FM_EXTRACT_SAMPLE; }
    }
    const u64 o = out_off[q];  // position x of the string is cell o + x - f
    InvStage<CellT> sg{out, o * sizeof(CellT), (o + e - f) * sizeof(CellT)};
    for (; p > f; p--) {  // p - f steps: L_k - f on the walk, fewer than e - f + FM_EXTRACT_SAMPLE from a sample
        const u64 x = ld_gather8(E + r);
        if (p <= e) sg.put(o + (p - 1 - f), inv_sym(x));
        r = inv_lf(x);
    }
    sg.flush();
}

// ---- LCP (DESIGN.md §12, "LCP"): row j's suffix is S_k[p .. L_k) $_k, string k occupies T[o_k .. o_k + L_k] with o_k = off[k] + k
// (off = exclusive scan of L), its separator last; a separator cell never matches ----
// walk path: string k from row k (position L_k) down to position 0, writing SA of every row it meets and its cells of T
static __global__ void __launch_bounds__(INV_THREADS) fm_lcp_walk_kernel(const u64* __restrict__ E, u32 N, u32 sep, const u32* __restrict__ len, const u32* __restrict__ off,
                                                                         u32* __restrict__ SA, u32* __restrict__ T) {
    const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N) return;
    const u32 L = len[k], o = off[k] + k;
    InvStage<u32> sg{(u8*)T, (u64)o * 4, ((u64)o + L + 1) * 4};
    sg.put((u64)o + L, sep);
    SA[k] = o + L;
    u32 r = k;
    for (u32 p = L; p > 0; p--) {  // L steps, counted by the count pass
        const u64 e = ld_gather8(E + r);
        r = inv_lf(e);
        sg.put((u64)o + p - 1, inv_sym(e));  // the row at position p holds S_k[p - 1]
        SA[r] = o + p - 1;
    }
    sg.flush();
}
// table path: L_k = the offset of row k < N ($_k) in the locate table
static __global__ void __launch_bounds__(INV_THREADS) fm_lcp_len_kernel(const u64* __restrict__ doc, u32 N, u32* __restrict__ len) {
    const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < N) len[k] = (u32)doc[k];
}
// table path: one thread per row, (k, p) from the locate table
static __global__ void __launch_bounds__(INV_THREADS) fm_lcp_table_kernel(const u64* __restrict__ E, const u64* __restrict__ doc, u32 n, u32 N, u32 sep,
                                                                          const u32* __restrict__ off, u32* __restrict__ SA, u32* __restrict__ T) {
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const u64 t = doc[j];
    const u32 k = (u32)(t >> 32), p = (u32)t, i = ld_gather4(off + k) + k + p;
    SA[j] = i;
    if (p) T[i - 1] = inv_sym(E[j]);
    if (j < N) T[i] = sep;
}
// irreducible rows: j >= N whose BWT symbol is the separator or differs from row j - 1's, one bit each (bits[j / 32]); every other
// row j >= N has LCP[LF(j)] = 1 + LCP[j]. The rows j < N ($_k) store PLCP 0 as a[SA[j]] = SA[j] (a is zero on entry).
static __global__ void __launch_bounds__(INV_THREADS) fm_lcp_flags_kernel(const u64* __restrict__ E, const u32* __restrict__ SA, u32 n, u32 N, u32 sep, u32* __restrict__ bits,
                                                                          u32* __restrict__ a) {
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    bool irr = false;
    if (j < N) {
        const u32 i = SA[j];
        a[i] = i;
    } else if (j < n) {
        const u32 c = inv_sym(E[j]);
        irr = c == sep || c != inv_sym(E[j - 1]);
    }
    const u32 m = __ballot_sync(0xffffffffu, irr);
    if (lane_id() == 0 && j < n) bits[j >> 5] = m;
}
// one warp per irreducible row j (grid-stride): LCE of T[SA[j] ..] and T[SA[j - 1] ..], 32 cells a step, the first mismatch or
// separator found by a ballot; a[SA[j]] = LCE + SA[j]; the LCEs summed into *sum, one atomic per warp
static __global__ void __launch_bounds__(INV_THREADS) fm_lcp_lce_kernel(const u32* __restrict__ rows, u64 n_rows, const u32* __restrict__ SA, const u32* __restrict__ T, u32 n,
                                                                        u32 sep, u32* __restrict__ a, u64* sum) {
    const u32 lane = lane_id();
    const u64 warps = ((u64)gridDim.x * blockDim.x) >> 5;
    u64 tot = 0;
    for (u64 w = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_rows; w += warps) {  // warp-uniform
        const u32 j = rows[w], x = SA[j], y = SA[j - 1];
        u32 l = 0;
        for (;;) {  // both strings end in a separator: at most min of their remaining lengths / 32 + 1 steps
            const u32 px = x + l + lane, py = y + l + lane;  // x + l, y + l < n < 2^32 - 16 while the loop runs
            const u32 cx = px < n ? T[px] : sep, cy = py < n ? T[py] : sep;
            const u32 stop = __ballot_sync(0xffffffffu, cx != cy || cx == sep);
            if (stop) { l += __ffs(stop) - 1; break; }
            l += 32;
        }
        if (lane == 0) a[x] = x + l;
        tot += l;
    }
    if (lane == 0 && tot) atomicAdd(sum, tot);
}
// M[i + 1] = max(a[0 .. i]) = PLCP[i] + i: LCP[j] = PLCP[SA[j]] for j >= N, 0 below
static __global__ void __launch_bounds__(INV_THREADS) fm_lcp_gather_kernel(const u32* __restrict__ SA, const u32* __restrict__ M, u32 n, u32 N, u32* __restrict__ lcp) {
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    if (j < N) { lcp[j] = 0; return; }
    const u32 i = SA[j];
    lcp[j] = ld_gather4(M + i + 1) - i;
}

inline FmView fm_view(const FmIndex& x) {
    return FmView{x.t.start.p, x.t.sym.p, x.t.len.p, x.t.F.p, x.t.order.p, x.dir_sym.p, x.dir_first.p, x.dir_C.p, (u32)x.t.n, (u32)x.t.n_runs, (u32)x.n_dir, x.t.sep};
}

// Load of a checked image (as lf_table_build) into the context's index; the index already loaded was dropped by the caller.
inline void fm_load(grlgpu_ctx* c, const u8* image, u64 image_bytes, grlgpu_fm_t* info) {
    cudaStream_t st = c->st;
    Timer t_all(st);
    t_all.start();
    std::unique_ptr<FmIndex> x(new FmIndex());
    LfTable& t = x->t;
    DevBuf<u32> keys;
    lf_table_build(image, image_bytes, t, &keys, st, "FM-index load on the device");
    const u32 n = (u32)t.n, nr = (u32)t.n_runs;
    if (n) {
        {   // directory: one entry per distinct symbol of the sorted keys
            DevBuf<u32> flags(nr, st), excl((u64)nr + 1, st);
            GRL_LAUNCH("ind_head_flags", (u64)nr * 8, ind_head_flags_kernel, grid_for(nr, 256), 256, 0, st, keys.p, nr, flags.p);
            x->n_dir = ind_scan_total(flags.p, excl.p, nr, st);
            x->dir_sym.alloc(x->n_dir, st);
            x->dir_first.alloc(x->n_dir + 1, st);
            x->dir_C.alloc(x->n_dir, st);
            GRL_LAUNCH("ind_compact_runs", (u64)nr * 16, ind_compact_runs_kernel, grid_for(nr, 256), 256, 0, st, keys.p, (const u32*)nullptr, flags.p, excl.p, nr, nr,
                       (u32)x->n_dir, x->dir_sym.p, x->dir_first.p);
            GRL_LAUNCH("fm_dir_c", x->n_dir * 12 + x->n_dir * 64, fm_dir_c_kernel, grid_for(x->n_dir, INV_THREADS), INV_THREADS, 0, st, x->dir_first.p, t.order.p, t.F.p,
                       (u32)x->n_dir, x->dir_C.p);
        }
        keys.release();
        x->psi.alloc(n, st);
        GRL_LAUNCH("fm_psi", (u64)n * (8 + 32), fm_psi_kernel, grid_for(n, INV_THREADS), INV_THREADS, 0, st, t.E.p, n, x->psi.p);
    }
    t_all.stop();
    info->n = t.n;
    info->n_strings = t.N;
    info->n_runs = t.n_runs;
    info->sigma = x->n_dir;
    info->sep = t.sep;
    info->load_ms = t_all.ms();  // synchronises the stream
    c->fm = std::move(x);
}

// the locate table of the loaded index (once): pointer jumping over LF, then one entry per row; error messages start with `who`
inline u32 fm_build_doc(FmIndex& x, u32* flag, cudaStream_t st, const char* who) {
    const u32 n = (u32)x.t.n, N = (u32)x.t.N;
    DevBuf<u64> P(n, st);
    DevBuf<u32> owner(n, st);
    const u32 rounds = inv_jump_converge(x.t.E.p, n, x.t.sep, P, owner.p, flag, st, who);
    {
        DevBuf<u32> slen(N, st);
        GRL_LAUNCH("inv_jump_owner", (u64)N * (8 + 4 + 32), inv_jump_owner_kernel, grid_for(N, INV_THREADS), INV_THREADS, 0, st, P.p, N, slen.p, owner.p);
    }
    x.doc.alloc(n, st);
    GRL_CUDA(cudaMemsetAsync(flag, 0, 4, st));
    GRL_LAUNCH("fm_doc", (u64)n * (8 + 32 + 32 + 8), fm_doc_kernel, grid_for(n, INV_THREADS), INV_THREADS, 0, st, x.t.E.p, P.p, owner.p, n, N, x.t.sep, x.doc.p, flag);
    if (d2h_scalar(flag, st)) {
        x.doc.release();
        throw Error(GRLGPU_ERR_ILL_FORMED, std::string(who) + ": a chain ends on a row that is not a string's separator row (an LF cycle without separator)");
    }
    x.doc_ready = true;
    return rounds;
}

// locate of every row of n_iv > 0 device intervals d_se (sp, ep per interval): d_occ receives the n_iv + 1 occurrence offsets, d_id /
// d_pos the occurrences, interval by interval in row order; info->n_occ, path and jump_rounds are set. Errors: GRLGPU_ERR_ARG when
// cap_occ < n_occ (info->n_occ holds the number needed), GRLGPU_ERR_ILL_FORMED on an LF cycle without separator.
template <class Info>
u64 fm_locate_rows(grlgpu_ctx* c, const u64* d_se, u64 n_iv, u64 cap_occ, DevBuf<u64>& d_occ, DevBuf<u32>& d_id, DevBuf<u32>& d_pos, Timer& t_loc, Info* info) {
    cudaStream_t st = c->st;
    FmIndex& x = *c->fm;
    d_occ.alloc(n_iv + 1, st);
    {
        DevBuf<u64> cnt(n_iv, st);
        GRL_LAUNCH("fm_occ_count", n_iv * 24, fm_occ_count_kernel, grid_for(n_iv, INV_THREADS), INV_THREADS, 0, st, d_se, n_iv, cnt.p);
        exclusive_scan<u64, u64>(cnt.p, d_occ.p, n_iv, d_occ.p + n_iv, st);
    }
    const u64 n_occ = d2h_scalar(d_occ.p + n_iv, st);
    info->n_occ = n_occ;
    if (n_occ > cap_occ) throw Error(GRLGPU_ERR_ARG, "locate: the occurrences need a capacity of " + std::to_string(n_occ));
    t_loc.start();
    d_id.alloc(n_occ, st);
    d_pos.alloc(n_occ, st);
    DevBuf<u32> flag(1, st);
    const bool force_walk = (c->flags & GRLGPU_FLAG_FORCE_WALK) != 0, force_jump = (c->flags & GRLGPU_FLAG_FORCE_JUMP) != 0 && !force_walk;
    bool walk = n_occ && !force_jump && (force_walk || !x.doc_ready);  // once built, the table answers every call
    if (walk) {  // rows off a cycle reach a separator row within n LF steps and a row < N within n psi steps: the bound n never overflows
        const u64 B = force_walk ? x.t.n : inv_walk_bound(x.t.n);
        flag.zero();
        GRL_LAUNCH("fm_locate_walk", n_occ * (8 + 8 + 8 * 2) + (u64)n_occ * 32 * 16, fm_locate_walk_kernel, grid_for(n_occ, INV_THREADS), INV_THREADS, 0, st, x.t.E.p, x.psi.p,
                   (u32)x.t.N, x.t.sep, d_se, d_occ.p, n_iv, n_occ, (u32)B, d_id.p, d_pos.p, flag.p);
        if (d2h_scalar(flag.p, st)) {
            if (force_walk) throw Error(GRLGPU_ERR_ILL_FORMED, "locate: a walk of n steps met no separator (an LF cycle without separator)");
            walk = false;
        }
    }
    info->path = (walk || !n_occ) ? 0 : 1;
    if (n_occ && !walk) {
        if (!x.doc_ready) info->jump_rounds = fm_build_doc(x, flag.p, st, "locate");
        GRL_LAUNCH("fm_locate_table", n_occ * (8 + 8 + 8 + 32), fm_locate_table_kernel, grid_for(n_occ, INV_THREADS), INV_THREADS, 0, st, x.doc.p, d_se, d_occ.p, n_iv, n_occ,
                   d_id.p, d_pos.p);
    }
    t_loc.stop();
    return n_occ;
}

// count (str_id == nullptr) or locate of n_pat > 0 checked patterns on the loaded index
inline void fm_query(grlgpu_ctx* c, const void* pat, const uint64_t* pat_off, u64 n_pat, int pat_bytes, uint64_t* sp_ep, uint64_t* occ_off, u32* str_id, u32* str_pos, u64 cap_occ,
                     grlgpu_fm_query_t* info) {
    cudaStream_t st = c->st;
    FmIndex& x = *c->fm;
    const u64 n_syms = pat_off[n_pat];
    info->n_pat = n_pat;
    info->n_pat_syms = n_syms;
    const bool locate = str_id != nullptr || occ_off != nullptr;
    Timer t_all(st), t_search(st), t_loc(st);
    t_all.start();
    t_search.start();
    DevBuf<u64> d_se(2 * n_pat, st);
    if (x.t.n == 0) d_se.zero();  // no rows: every interval is empty
    else {
        DevBuf<u8> d_pat(n_syms * pat_bytes, st);
        DevBuf<u64> d_off(n_pat + 1, st);
        GRL_CUDA(cudaMemcpyAsync(d_pat.p, pat, n_syms * pat_bytes, cudaMemcpyHostToDevice, st));
        GRL_CUDA(cudaMemcpyAsync(d_off.p, pat_off, (n_pat + 1) * 8, cudaMemcpyHostToDevice, st));
        const FmView v = fm_view(x);
        // per pattern symbol two searches over the run starts and one over its slice: one 32 B sector per probe
        const u64 model = n_pat * 24 + n_syms * (pat_bytes + 2 * 64 * 32);
        switch (pat_bytes) {
            case 1: GRL_LAUNCH("fm_count", model, (fm_count_kernel<u8>), grid_for(n_pat, INV_THREADS), INV_THREADS, 0, st, v, (const u8*)d_pat.p, d_off.p, n_pat, d_se.p); break;
            case 2: GRL_LAUNCH("fm_count", model, (fm_count_kernel<u16>), grid_for(n_pat, INV_THREADS), INV_THREADS, 0, st, v, (const u16*)d_pat.p, d_off.p, n_pat, d_se.p); break;
            case 4: GRL_LAUNCH("fm_count", model, (fm_count_kernel<u32>), grid_for(n_pat, INV_THREADS), INV_THREADS, 0, st, v, (const u32*)d_pat.p, d_off.p, n_pat, d_se.p); break;
            default: GRL_LAUNCH("fm_count", model, (fm_count_kernel<u64>), grid_for(n_pat, INV_THREADS), INV_THREADS, 0, st, v, (const u64*)d_pat.p, d_off.p, n_pat, d_se.p); break;
        }
    }
    t_search.stop();
    if (!locate) {
        GRL_CUDA(cudaMemcpyAsync(sp_ep, d_se.p, 2 * n_pat * 8, cudaMemcpyDeviceToHost, st));
        t_all.stop();
        info->search_ms = t_search.ms();
        info->device_ms = t_all.ms();  // waits for the copy
        return;
    }
    DevBuf<u64> d_occ;
    DevBuf<u32> d_id, d_pos;
    const u64 n_occ = fm_locate_rows(c, d_se.p, n_pat, cap_occ, d_occ, d_id, d_pos, t_loc, info);
    GRL_CUDA(cudaMemcpyAsync(occ_off, d_occ.p, (n_pat + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (n_occ) {
        GRL_CUDA(cudaMemcpyAsync(str_id, d_id.p, n_occ * 4, cudaMemcpyDeviceToHost, st));
        GRL_CUDA(cudaMemcpyAsync(str_pos, d_pos.p, n_occ * 4, cudaMemcpyDeviceToHost, st));
    }
    t_all.stop();
    info->search_ms = t_search.ms();
    info->locate_ms = t_loc.ms();
    info->device_ms = t_all.ms();  // waits for the copies
}

// the extract samples of the loaded index (once), from its locate table
inline void fm_build_samples(FmIndex& x, cudaStream_t st) {
    const u32 n = (u32)x.t.n, N = (u32)x.t.N;
    x.samp_off.alloc((u64)N + 1, st);
    GRL_LAUNCH("fm_samp_len", (u64)N * (8 + 4), fm_samp_len_kernel, grid_for(N, INV_THREADS), INV_THREADS, 0, st, x.doc.p, N, x.samp_off.p);
    exclusive_scan<u32, u32>(x.samp_off.p, x.samp_off.p, N, x.samp_off.p + N, st);
    const u32 n_samp = d2h_scalar(x.samp_off.p + N, st);  // at most n / S + N
    x.samp.alloc(n_samp, st);
    GRL_LAUNCH("fm_samp_fill", (u64)n * 8 + (u64)n_samp * (32 + 32), fm_samp_fill_kernel, grid_for(n, INV_THREADS), INV_THREADS, 0, st, x.doc.p, n, x.samp_off.p, x.samp.p);
    x.samp_ready = true;
}

template <class CellT>
void fm_extract_write(const FmIndex& x, const u32* id, const u32* from, const u32* len, const u32* Lq, const u64* off, u32 n_req, bool samples, u8* out, u64 steps,
                      u64 n_cells, cudaStream_t st) {
    GRL_LAUNCH("fm_extract_write", (u64)n_req * (4 * 4 + 8) + steps * 32 + n_cells * sizeof(CellT), (fm_extract_write_kernel<CellT>), grid_for(n_req, INV_THREADS), INV_THREADS, 0, st,
               x.t.E.p, id, from, len, Lq, off, n_req, samples ? x.samp.p : nullptr, samples ? x.samp_off.p : nullptr, out);
}

// extract of 0 < n_req < 2^32 checked requests (every str_id < N) on the loaded index
inline void fm_extract(grlgpu_ctx* c, const u32* str_id, const u32* from, const u32* len, u32 n_req, int w, uint64_t* out_off, void* out, u64 cap_cells,
                       grlgpu_fm_extract_t* info) {
    cudaStream_t st = c->st;
    FmIndex& x = *c->fm;
    const u64 n = x.t.n, N = x.t.N, mean_len = (n - N) / N;  // N >= 1: some request names a string
    info->n_req = n_req;
    Timer t_all(st), t_ext(st);
    t_all.start();
    DevBuf<u32> d_req(3 * (u64)n_req, st);
    u32 *d_id = d_req.p, *d_from = d_id + n_req, *d_len = d_from + n_req;
    GRL_CUDA(cudaMemcpyAsync(d_id, str_id, (u64)n_req * 4, cudaMemcpyHostToDevice, st));
    GRL_CUDA(cudaMemcpyAsync(d_from, from, (u64)n_req * 4, cudaMemcpyHostToDevice, st));
    GRL_CUDA(cudaMemcpyAsync(d_len, len, (u64)n_req * 4, cudaMemcpyHostToDevice, st));
    t_ext.start();
    DevBuf<u32> Lq(n_req, st), flag(1, st);
    const bool force_walk = (c->flags & GRLGPU_FLAG_FORCE_WALK) != 0, force_jump = (c->flags & GRLGPU_FLAG_FORCE_JUMP) != 0 && !force_walk;
    bool walk = !force_jump && (force_walk || !(x.doc_ready || x.samp_ready));  // once the samples or the locate table exist, they answer
    if (walk) {  // a walk from row k ends within n steps (the LF cycle of k holds the separator row LF^-1(k)): the bound n never overflows
        const u64 B = force_walk ? n : inv_walk_bound(n);
        flag.zero();
        GRL_LAUNCH("inv_walk_count", (u64)n_req * (8 + mean_len * 32), inv_walk_count_kernel, grid_for(n_req, INV_THREADS), INV_THREADS, 0, st, x.t.E.p, (const u32*)d_id, n_req,
                   x.t.sep, (u32)B, Lq.p, flag.p);
        walk = d2h_scalar(flag.p, st) == 0;
    }
    info->path = walk ? 0 : 1;
    if (!walk) {
        if (!x.doc_ready) info->jump_rounds = fm_build_doc(x, flag.p, st, "extract");
        if (!x.samp_ready) fm_build_samples(x, st);
    }
    DevBuf<u64> d_off((u64)n_req + 1, st);
    {
        DevBuf<u64> cnt(n_req, st);
        GRL_LAUNCH("fm_extract_size", (u64)n_req * (4 * 4 + 8) + (walk ? 0 : (u64)n_req * 32), fm_extract_size_kernel, grid_for(n_req, INV_THREADS), INV_THREADS, 0, st, d_id, d_from,
                   d_len, n_req, walk ? (const u64*)nullptr : x.doc.p, Lq.p, cnt.p);
        exclusive_scan<u64, u64>(cnt.p, d_off.p, n_req, d_off.p + n_req, st);
    }
    const u64 n_cells = d2h_scalar(d_off.p + n_req, st);
    info->n_cells = n_cells;
    if (n_cells > cap_cells) {  // the times of the work done so far (a sizing call may have built the locate table and the samples)
        t_ext.stop();
        t_all.stop();
        info->extract_ms = t_ext.ms();
        info->device_ms = t_all.ms();
        throw Error(GRLGPU_ERR_ARG, "extract: the cells need a capacity of " + std::to_string(n_cells));
    }
    DevBuf<u8> dout(n_cells * w + 16, st);
    // steps of the model: the walk goes from each string's end (mean length), a sample at most S - 1 positions past e (S / 2 on average)
    const u64 steps = walk ? (u64)n_req * mean_len : n_cells + (u64)n_req * FM_EXTRACT_SAMPLE / 2;
    switch (w) {
        case 1: fm_extract_write<u8>(x, d_id, d_from, d_len, Lq.p, d_off.p, n_req, !walk, dout.p, steps, n_cells, st); break;
        case 2: fm_extract_write<u16>(x, d_id, d_from, d_len, Lq.p, d_off.p, n_req, !walk, dout.p, steps, n_cells, st); break;
        case 4: fm_extract_write<u32>(x, d_id, d_from, d_len, Lq.p, d_off.p, n_req, !walk, dout.p, steps, n_cells, st); break;
        default: fm_extract_write<u64>(x, d_id, d_from, d_len, Lq.p, d_off.p, n_req, !walk, dout.p, steps, n_cells, st); break;
    }
    t_ext.stop();
    GRL_CUDA(cudaMemcpyAsync(out_off, d_off.p, ((u64)n_req + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (n_cells) GRL_CUDA(cudaMemcpyAsync(out, dout.p, n_cells * w, cudaMemcpyDeviceToHost, st));
    t_all.stop();
    info->extract_ms = t_ext.ms();
    info->device_ms = t_all.ms();  // waits for the copies
}

// approximate search: the first pool holds max(FM_APPROX_POOL_MIN, 4 n_pat) hits; a search that finds more runs once more with
// the exact size. 20 bytes per pool entry, 12 more per hit for the sort.
constexpr u64 FM_APPROX_POOL_MIN = 1ull << 16;

// backtracking search of 0 < n_pat < 2^32 checked patterns with at most kmax substitutions: the hits in (pattern, sp) order in
// d_se (sp, ep per hit) and d_mm (d per hit), per-pattern hit offsets in d_hoff (n_pat + 1); info->n_pat(_syms), n_hits and n_lf
// are set. Returns the number of hits (GRLGPU_ERR_LIMIT from 2^32 hits).
inline u64 fm_approx_search(grlgpu_ctx* c, const void* pat, const uint64_t* pat_off, u64 n_pat, int pat_bytes, u32 kmax, DevBuf<u64>& d_se, DevBuf<u8>& d_mm,
                            DevBuf<u64>& d_hoff, grlgpu_fm_approx_t* info) {
    cudaStream_t st = c->st;
    FmIndex& x = *c->fm;
    const u64 n_syms = pat_off[n_pat];
    info->n_pat = n_pat;
    info->n_pat_syms = n_syms;
    d_hoff.alloc(n_pat + 1, st);
    if (x.t.n == 0) {  // no rows: no hits
        d_hoff.zero();
        return 0;
    }
    DevBuf<u8> d_pat(n_syms * pat_bytes, st);
    DevBuf<u64> d_off(n_pat + 1, st), cnt(n_pat, st), counters(2, st);
    GRL_CUDA(cudaMemcpyAsync(d_pat.p, pat, n_syms * pat_bytes, cudaMemcpyHostToDevice, st));
    GRL_CUDA(cudaMemcpyAsync(d_off.p, pat_off, (n_pat + 1) * 8, cudaMemcpyHostToDevice, st));
    const FmView v = fm_view(x);
    DevBuf<u64> key, ep_d;
    DevBuf<u32> slot;
    u64 cap = std::max(FM_APPROX_POOL_MIN, 4 * n_pat), h[2] = {0, 0};
    for (int pass = 0; pass < 2; pass++) {  // the second pass only when the first pool was too small, with the exact size
        key.alloc(cap, st);
        ep_d.alloc(cap, st);
        slot.alloc(cap, st);
        counters.zero();
        // bytes known only from the LF_c count read back below: added to this launch's record then
        switch (pat_bytes) {
            case 1: GRL_LAUNCH("fm_approx", 0, (fm_approx_kernel<u8>), grid_for(n_pat, INV_THREADS), INV_THREADS, 0, st, v, (const u8*)d_pat.p, d_off.p, n_pat, kmax, cap, key.p, slot.p, ep_d.p, cnt.p, counters.p); break;
            case 2: GRL_LAUNCH("fm_approx", 0, (fm_approx_kernel<u16>), grid_for(n_pat, INV_THREADS), INV_THREADS, 0, st, v, (const u16*)d_pat.p, d_off.p, n_pat, kmax, cap, key.p, slot.p, ep_d.p, cnt.p, counters.p); break;
            case 4: GRL_LAUNCH("fm_approx", 0, (fm_approx_kernel<u32>), grid_for(n_pat, INV_THREADS), INV_THREADS, 0, st, v, (const u32*)d_pat.p, d_off.p, n_pat, kmax, cap, key.p, slot.p, ep_d.p, cnt.p, counters.p); break;
            default: GRL_LAUNCH("fm_approx", 0, (fm_approx_kernel<u64>), grid_for(n_pat, INV_THREADS), INV_THREADS, 0, st, v, (const u64*)d_pat.p, d_off.p, n_pat, kmax, cap, key.p, slot.p, ep_d.p, cnt.p, counters.p); break;
        }
        d2h_small(h, counters.p, sizeof(h), st);
        // per LF_c evaluation two binary searches (run starts, c's slice), one 32 B sector per probe, as fm_count; the hits' stores
        if (g_prof && g_prof->timing && !g_prof->pending.empty()) g_prof->pending.back().bytes = n_pat * 24 + n_syms * pat_bytes + h[1] * 64 * 32 + std::min(h[0], cap) * 20;
        if (h[0] >> 32) throw Error(GRLGPU_ERR_LIMIT, "approximate search: 2^32 hits or more");
        if (h[0] <= cap) break;
        cap = h[0];
    }
    const u64 n_hits = h[0];
    info->n_hits = n_hits;
    info->n_lf = h[1];
    exclusive_scan<u64, u64>(cnt.p, d_hoff.p, n_pat, d_hoff.p + n_pat, st);
    {
        DevBuf<u64> key_alt(n_hits, st);
        DevBuf<u32> slot_alt(n_hits, st);
        u64 *kp = key.p, *ka = key_alt.p;
        u32 *vp = slot.p, *va = slot_alt.p;
        radix_sort_pairs(&kp, &vp, &ka, &va, n_hits, 32 + bit_width64(n_pat - 1), st);
        d_se.alloc(2 * n_hits, st);
        d_mm.alloc(n_hits, st);
        GRL_LAUNCH("fm_approx_gather", n_hits * (8 + 4 + 32 + 16 + 1), fm_approx_gather_kernel, grid_for(n_hits, INV_THREADS), INV_THREADS, 0, st, kp, vp, ep_d.p, n_hits, d_se.p, d_mm.p);
    }
    return n_hits;
}

// approximate count: the hits of 0 < n_pat < 2^32 checked patterns with at most kmax substitutions
inline void fm_approx_count(grlgpu_ctx* c, const void* pat, const uint64_t* pat_off, u64 n_pat, int pat_bytes, u32 kmax, uint64_t* hit_off, uint64_t* sp_ep, uint8_t* hit_mm,
                            u64 cap_hits, grlgpu_fm_approx_t* info) {
    cudaStream_t st = c->st;
    Timer t_all(st), t_search(st);
    t_all.start();
    t_search.start();
    DevBuf<u64> d_se, d_hoff;
    DevBuf<u8> d_mm;
    const u64 n_hits = fm_approx_search(c, pat, pat_off, n_pat, pat_bytes, kmax, d_se, d_mm, d_hoff, info);
    t_search.stop();
    if (n_hits > cap_hits) {  // the times of the search already run
        t_all.stop();
        info->search_ms = t_search.ms();
        info->device_ms = t_all.ms();
        throw Error(GRLGPU_ERR_ARG, "approximate count: the hits need a capacity of " + std::to_string(n_hits));
    }
    GRL_CUDA(cudaMemcpyAsync(hit_off, d_hoff.p, (n_pat + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (n_hits) {
        GRL_CUDA(cudaMemcpyAsync(sp_ep, d_se.p, 2 * n_hits * 8, cudaMemcpyDeviceToHost, st));
        GRL_CUDA(cudaMemcpyAsync(hit_mm, d_mm.p, n_hits, cudaMemcpyDeviceToHost, st));
    }
    t_all.stop();
    info->search_ms = t_search.ms();
    info->device_ms = t_all.ms();  // waits for the copies
    for (u64 i = 0; i < n_hits; i++) info->n_occ += sp_ep[2 * i + 1] - sp_ep[2 * i];
}

// approximate locate: every occurrence of every hit, with the d of its hit; pattern q's occurrences in row order
inline void fm_approx_locate(grlgpu_ctx* c, const void* pat, const uint64_t* pat_off, u64 n_pat, int pat_bytes, u32 kmax, uint64_t* occ_off, u32* str_id, u32* str_pos,
                             uint8_t* occ_mm, u64 cap_occ, grlgpu_fm_approx_t* info) {
    cudaStream_t st = c->st;
    Timer t_all(st), t_search(st), t_loc(st);
    t_all.start();
    t_search.start();
    DevBuf<u64> d_se, d_hoff;
    DevBuf<u8> d_mm;
    const u64 n_hits = fm_approx_search(c, pat, pat_off, n_pat, pat_bytes, kmax, d_se, d_mm, d_hoff, info);
    t_search.stop();
    if (n_hits == 0) {
        memset(occ_off, 0, (n_pat + 1) * 8);
        t_all.stop();
        info->search_ms = t_search.ms();
        info->device_ms = t_all.ms();
        return;
    }
    DevBuf<u64> d_occ;
    DevBuf<u32> d_id, d_pos;
    const u64 n_occ = fm_locate_rows(c, d_se.p, n_hits, cap_occ, d_occ, d_id, d_pos, t_loc, info);
    DevBuf<u8> d_omm(n_occ, st);
    DevBuf<u64> d_qoff(n_pat + 1, st);
    GRL_LAUNCH("fm_approx_occ_mm", n_occ * (1 + 32 * 2) + n_hits, fm_approx_occ_mm_kernel, grid_for(n_occ, INV_THREADS), INV_THREADS, 0, st, d_occ.p, n_hits, d_mm.p, n_occ, d_omm.p);
    GRL_LAUNCH("fm_approx_occ_off", (n_pat + 1) * (8 + 32 + 8), fm_approx_occ_off_kernel, grid_for(n_pat + 1, INV_THREADS), INV_THREADS, 0, st, d_occ.p, d_hoff.p, n_pat, d_qoff.p);
    GRL_CUDA(cudaMemcpyAsync(occ_off, d_qoff.p, (n_pat + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (n_occ) {
        GRL_CUDA(cudaMemcpyAsync(str_id, d_id.p, n_occ * 4, cudaMemcpyDeviceToHost, st));
        GRL_CUDA(cudaMemcpyAsync(str_pos, d_pos.p, n_occ * 4, cudaMemcpyDeviceToHost, st));
        GRL_CUDA(cudaMemcpyAsync(occ_mm, d_omm.p, n_occ, cudaMemcpyDeviceToHost, st));
    }
    t_all.stop();
    info->search_ms = t_search.ms();
    info->locate_ms = t_loc.ms();
    info->device_ms = t_all.ms();  // waits for the copies
}

// LCP of every row of the loaded index (n > 0) into the host array lcp (n entries, checked by the caller)
inline void fm_lcp(grlgpu_ctx* c, u32* lcp, grlgpu_fm_lcp_t* info) {
    cudaStream_t st = c->st;
    FmIndex& x = *c->fm;
    const u32 n = (u32)x.t.n, N = (u32)x.t.N, sep = x.t.sep;
    Timer t_all(st), t_sa(st), t_lcp(st);
    t_all.start();
    t_sa.start();
    // ---- 1: SA and T (T holds n + 1 cells: it receives the max-scan of step 4) ----
    DevBuf<u32> SA(n, st), T((u64)n + 1, st), a((u64)n + 1, st), flag(1, st);
    {
        DevBuf<u32> len(N, st), off((u64)N + 1, st);
        const bool force_walk = (c->flags & GRLGPU_FLAG_FORCE_WALK) != 0, force_jump = (c->flags & GRLGPU_FLAG_FORCE_JUMP) != 0 && !force_walk;
        bool walk = !force_jump && (force_walk || !x.doc_ready);  // once built, the locate table answers
        if (walk) {  // a walk from row k ends within n steps: the bound n never overflows
            const u64 B = force_walk ? n : inv_walk_bound(n);
            flag.zero();
            GRL_LAUNCH("inv_walk_count", (u64)N * 4 + (u64)(n - N) * 32, inv_walk_count_kernel, grid_for(N, INV_THREADS), INV_THREADS, 0, st, x.t.E.p, (const u32*)nullptr, N, sep,
                       (u32)B, len.p, flag.p);
            walk = d2h_scalar(flag.p, st) == 0;
        }
        info->path = walk ? 0 : 1;
        if (walk) {
            exclusive_scan<u32, u32>(len.p, off.p, N, off.p + N, st);
            if ((u64)d2h_scalar(off.p + N, st) + N != n) throw Error(GRLGPU_ERR_ILL_FORMED, "lcp: the strings do not cover the BWT (an LF cycle without separator)");
            GRL_LAUNCH("fm_lcp_walk", (u64)N * 8 + (u64)n * (32 + 32 + 4), fm_lcp_walk_kernel, grid_for(N, INV_THREADS), INV_THREADS, 0, st, x.t.E.p, N, sep, len.p, off.p, SA.p, T.p);
        } else {
            if (!x.doc_ready) info->jump_rounds = fm_build_doc(x, flag.p, st, "lcp");
            GRL_LAUNCH("fm_lcp_len", (u64)N * (8 + 4), fm_lcp_len_kernel, grid_for(N, INV_THREADS), INV_THREADS, 0, st, x.doc.p, N, len.p);
            exclusive_scan<u32, u32>(len.p, off.p, N, off.p + N, st);
            GRL_LAUNCH("fm_lcp_table", (u64)n * (8 + 8 + 4 + 32 + 32) + (u64)N * 32, fm_lcp_table_kernel, grid_for(n, INV_THREADS), INV_THREADS, 0, st, x.t.E.p, x.doc.p, n, N,
                       sep, off.p, SA.p, T.p);
        }
    }
    t_sa.stop();
    t_lcp.start();
    // ---- 2: irreducible rows; the separator rows' PLCP 0 into a ----
    a.zero();
    DevBuf<u32> bits(div_up(n, 32), st), rows;
    GRL_LAUNCH("fm_lcp_flags", (u64)n * 8 + n / 8 + (u64)N * (4 + 32), fm_lcp_flags_kernel, grid_for(n, INV_THREADS), INV_THREADS, 0, st, x.t.E.p, SA.p, n, N, sep, bits.p, a.p);
    BitmapCompactor bc;
    const u64 n_irr = bc.count(bits.p, n, st);
    rows.alloc(n_irr, st);
    bc.write<u32>(nullptr, rows.p);
    bits.release();
    // ---- 3: one warp per irreducible row ----
    DevBuf<u64> sum(1, st);
    sum.zero();
    if (n_irr) {
        const u64 blocks = std::min<u64>(div_up(n_irr, INV_THREADS / 32), (u64)c->n_sm * (2048 / INV_THREADS));  // one wave of full SMs at most
        // bytes known only from the LCE sum read back below: added to this launch's record then
        GRL_LAUNCH("fm_lcp_lce", 0, fm_lcp_lce_kernel, (unsigned)blocks, INV_THREADS, 0, st, rows.p, n_irr, SA.p, T.p, n, sep, a.p, sum.p);
    }
    const u64 sum_irr = d2h_scalar(sum.p, st);
    // per row its index, two SA gathers, and per 32-cell step two 128 B segments of T; the a store
    if (n_irr && g_prof && g_prof->timing && !g_prof->pending.empty()) g_prof->pending.back().bytes = n_irr * (4 + 2 * 32 + 32) + (sum_irr / 32 + n_irr) * 2 * 128;
    info->n_irreducible = n_irr;
    info->sum_irreducible = sum_irr;
    rows.release();
    // ---- 4: inclusive max over text positions: T[i + 1] = max(a[0 .. i]) = PLCP[i] + i ----
    exclusive_scan<u32, u32, ScanMax>(a.p, T.p, (u64)n + 1, (u32*)nullptr, st);
    // ---- 5: back to rows, into a ----
    GRL_LAUNCH("fm_lcp_gather", (u64)n * (4 + 4) + (u64)(n - N) * 32, fm_lcp_gather_kernel, grid_for(n, INV_THREADS), INV_THREADS, 0, st, SA.p, T.p, n, N, a.p);
    t_lcp.stop();
    GRL_CUDA(cudaMemcpyAsync(lcp, a.p, (u64)n * 4, cudaMemcpyDeviceToHost, st));
    t_all.stop();
    info->sa_ms = t_sa.ms();
    info->lcp_ms = t_lcp.ms();
    info->device_ms = t_all.ms();  // waits for the copy
}
