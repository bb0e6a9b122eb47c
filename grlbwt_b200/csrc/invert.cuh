// Inversion of a BCR BWT ON THE DEVICE: the image of a .rl_bwt file back to the string collection, byte for byte what
// host/tools/reverse_bwt.cpp writes (reference scripts/reverse_bwt.cpp:5-54), without its host LF walk of O(log r) per step.
//   a  LF table      decode the records, run starts by a scan, each run's F position C[c] + before[k] by a stable sort of the
//                    run indices on the symbol and a scan of the lengths in that order; then one packed 8-byte entry per
//                    position, E[j] = {LF(j) << 32 | BWT[j]}: an LF step is one random 8-byte gather
//   b  walk          one thread per requested string follows its chain from row i (count pass, scan, write pass)
//   c  jumping       list ranking over the LF permutation (succ, distance) by pointer jumping, then one scatter per row
//   d  selection     the count pass of (b) runs with a step bound B; a chain longer than B switches to (c)
// Convention of reverse_bwt: the separator is the smallest symbol (of a non-empty record), there are N strings where N is its
// count, row i < N is the suffix $_i, and the chain from row i up to a row whose BWT symbol is the separator is string i
// backwards. LF built from any run list is a permutation that maps the separator rows onto [0, N), so that chain ends within
// n steps for every input; a run list that is not a BWT can still leave rows on cycles without a separator, which both paths
// detect. Positions and lengths are 32-bit (n < 0xfffffff0, symbols < 2^32): larger inputs are left to the host tool.
// Part a (lf_table_build), the walk bound, the count pass and pointer jumping (inv_jump_converge) are shared with the FM-index of fm.cuh.
// Included by grlgpu.cu inside its anonymous namespace.
#pragma once

constexpr int INV_THREADS = 256;
constexpr int INV_FILL_ITEMS = 8;
constexpr int INV_FILL_TILE = INV_THREADS * INV_FILL_ITEMS;
// selection: the walk keeps every chain of at most B steps, B = max(INV_B_MIN, n / INV_B_DIV) (DESIGN.md, "Inversion on the device")
constexpr u64 INV_B_MIN = 4096;
constexpr u64 INV_B_DIV = 2048;
constexpr u32 INV_NOT_SEP = 0xffffffffu;  // owner[] of a row whose BWT symbol is not the separator
constexpr u32 INV_UNREQ = 0xfffffffeu;    // owner[] of a separator row that ends no requested string

__device__ __forceinline__ u32 inv_sym(u64 e) { return (u32)e; }
__device__ __forceinline__ u32 inv_lf(u64 e) { return (u32)(e >> 32); }

// st[0]: a symbol or a length does not fit 32 bits; st[1]: largest symbol; st[2]: smallest symbol of a non-empty record
static __global__ void __launch_bounds__(INV_THREADS) inv_decode_kernel(const u8* __restrict__ rec, u64 n_runs, int sb, int fb, u32* __restrict__ sym,
                                                                        u32* __restrict__ len, u32* st) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u32 mx = 0, mn = 0xffffffffu, bad = 0;
    if (i < n_runs) {
        const u8* r = rec + i * (u64)(sb + fb);
        u64 s = 0, l = 0;
        for (int b = 0; b < sb; b++) s |= (u64)r[b] << (8 * b);       // sb <= 8 (checked on the host)
        for (int b = 0; b < fb; b++) l |= (u64)r[sb + b] << (8 * b);  // fb <= 8
        bad = (s >> 32) || (l >> 32);
        sym[i] = (u32)s;
        len[i] = (u32)l;
        mx = (u32)s;
        if (l) mn = (u32)s;
    }
    bad = __any_sync(0xffffffffu, bad);
    mx = warp_max(mx);
    mn = warp_min(mn);
    if (lane_id() == 0) {
        if (bad) atomicExch(&st[0], 1u);
        atomicMax(&st[1], mx);
        atomicMin(&st[2], mn);
    }
}
static __global__ void __launch_bounds__(INV_THREADS) inv_sep_count_kernel(const u32* __restrict__ sym, const u32* __restrict__ len, u64 n_runs, u32 sep, u64* cnt) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u64 c = (i < n_runs && sym[i] == sep) ? len[i] : 0;
    c = warp_sum(c);
    if (lane_id() == 0 && c) atomicAdd(cnt, c);
}
static __global__ void __launch_bounds__(INV_THREADS) inv_iota_kernel(u32* __restrict__ v, u64 n) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = (u32)i;
}
static __global__ void __launch_bounds__(INV_THREADS) inv_sorted_len_kernel(const u32* __restrict__ order, const u32* __restrict__ len, u64 n_runs, u32* __restrict__ slen) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n_runs) slen[k] = len[order[k]];
}
// fpos[k] = first F row of the k-th run in (symbol, run index) order = C[c] + before[k]
static __global__ void __launch_bounds__(INV_THREADS) inv_scatter_f_kernel(const u32* __restrict__ order, const u32* __restrict__ fpos, u64 n_runs, u32* __restrict__ F) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n_runs) F[order[k]] = fpos[k];
}
// E[j] = {LF(j), BWT[j]} for the CTA's tile of INV_FILL_TILE positions: one sorted search per CTA for the tile's run range,
// one per thread inside it for its first position, then a linear advance; stores go through shared memory, coalesced.
static __global__ void __launch_bounds__(INV_THREADS) inv_fill_kernel(const u32* __restrict__ start, const u32* __restrict__ F, const u32* __restrict__ sym, u32 n_runs,
                                                                      u32 n, u64* __restrict__ E) {
    __shared__ u64 stage[INV_FILL_TILE];
    __shared__ u32 k_range[2];
    const u32 j0 = blockIdx.x * INV_FILL_TILE;
    const u32 cnt = min((u32)INV_FILL_TILE, n - j0);
    // start[] has n_runs + 1 entries, start[n_runs] = n; the run holding j is the last one with start <= j (zero-length
    // records share their start with the next run and are never chosen)
    if (threadIdx.x == 0) {
        k_range[0] = ind_upper_bound(start, n_runs, j0) - 1;
        k_range[1] = ind_upper_bound(start, n_runs, j0 + cnt - 1) - 1;
    }
    __syncthreads();
    const u32 klo = k_range[0], khi = k_range[1];
    const u32 t0 = threadIdx.x * INV_FILL_ITEMS;
    if (t0 < cnt) {
        u32 k = klo + ind_upper_bound(start + klo, khi - klo + 1, j0 + t0) - 1;
#pragma unroll
        for (int q = 0; q < INV_FILL_ITEMS; q++) {
            const u32 t = t0 + q, j = j0 + t;
            if (t >= cnt) break;
            while (start[k + 1] <= j) k++;  // k only grows, and start[n_runs] = n > j: at most n_runs steps
            stage[t] = ((u64)(F[k] + (j - start[k])) << 32) | sym[k];
        }
    }
    __syncthreads();
    for (u32 t = threadIdx.x; t < cnt; t += INV_THREADS) E[(u64)j0 + t] = stage[t];
}

// ---- b: walk per string ----
// count pass: steps from row i to its separator row, at most `bound` (chains from rows < N end within n steps: bound >= n
// never overflows); more than `bound` raises *over and the caller switches to pointer jumping. Thread i walks string ids[i]
// (fm.cuh's extract), or string i when ids is null.
static __global__ void __launch_bounds__(INV_THREADS) inv_walk_count_kernel(const u64* __restrict__ E, const u32* __restrict__ ids, u32 n_req, u32 sep, u32 bound, u32* __restrict__ len,
                                                                            u32* over) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_req) return;
    u32 j = ids ? ids[i] : i;
    for (u32 t = 0; t < bound; t++) {  // bounded by `bound`
        const u64 e = ld_gather8(E + j);
        if (inv_sym(e) == sep) { len[i] = t; return; }
        j = inv_lf(e);
    }
    len[i] = bound;
    atomicExch(over, 1u);
}
// the cells of one string, written from its end backwards, leave the thread in aligned 16-byte blocks; the first and last
// block of a string may be shared with the neighbouring strings and are stored cell by cell
template <class CellT>
struct InvStage {
    u8* out;
    u64 lo_b, hi_b;  // bytes of this string: [lo_b, hi_b)
    u64 blk = ~0ull, w0 = 0, w1 = 0;
    __device__ void flush() {
        if (blk == ~0ull) return;
        const u64 b0 = blk * 16;
        if (b0 >= lo_b && b0 + 16 <= hi_b) {
            *reinterpret_cast<ulonglong2*>(out + b0) = make_ulonglong2(w0, w1);
            return;
        }
        for (u32 c = 0; c < 16 / sizeof(CellT); c++) {  // 16 / w cells per block
            const u64 a = b0 + c * sizeof(CellT);
            if (a < lo_b || a >= hi_b) continue;
            const u32 sh = c * sizeof(CellT) * 8;
            *reinterpret_cast<CellT*>(out + a) = (CellT)((sh < 64 ? w0 : w1) >> (sh & 63));
        }
    }
    __device__ void put(u64 cell, u64 v) {
        const u64 a = cell * sizeof(CellT);
        if ((a >> 4) != blk) { flush(); blk = a >> 4; w0 = w1 = 0; }
        const u32 sh = (u32)(a & 15) * 8;
        const u64 x = (u64)(CellT)v;  // the cell keeps the symbol's low bytes, as reverse_bwt's put_cell
        if (sh < 64) w0 |= x << sh; else w1 |= x << (sh - 64);
    }
};
template <class CellT>
__global__ void __launch_bounds__(INV_THREADS) inv_walk_write_kernel(const u64* __restrict__ E, u32 n_req, u32 sep, const u32* __restrict__ len, const u32* __restrict__ off,
                                                                     u8* __restrict__ out) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_req) return;
    const u32 L = len[i], o = off[i] + i;  // off = exclusive scan of the lengths: string i starts at off[i] + i
    InvStage<CellT> sg{out, (u64)o * sizeof(CellT), ((u64)o + L + 1) * sizeof(CellT)};
    sg.put((u64)o + L, sep);
    u32 j = i;
    for (u32 t = 0; t < L; t++) {  // L steps, counted by the count pass
        const u64 e = ld_gather8(E + j);
        sg.put((u64)o + L - 1 - t, inv_sym(e));
        j = inv_lf(e);
    }
    sg.flush();
}

// ---- c: pointer jumping over the LF permutation: P[j] = {d << 32 | succ} ----
static __global__ void __launch_bounds__(INV_THREADS) inv_jump_init_kernel(const u64* __restrict__ E, u32 n, u32 sep, u64* __restrict__ P, u32* __restrict__ owner) {
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const u64 e = E[j];
    const bool s = inv_sym(e) == sep;
    P[j] = s ? (u64)j : ((1ull << 32) | inv_lf(e));
    owner[j] = s ? INV_UNREQ : INV_NOT_SEP;
}
// one round: d[j] += d[succ[j]], succ[j] = succ[succ[j]]; *moved when some succ changed
static __global__ void __launch_bounds__(INV_THREADS) inv_jump_round_kernel(const u64* __restrict__ P, u32 n, u64* __restrict__ Q, u32* moved) {
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    bool mv = false;
    if (j < n) {
        const u64 p = P[j];
        const u32 s = (u32)p;
        const u64 q = ld_gather8(P + s);
        Q[j] = (((p >> 32) + (q >> 32)) << 32) | (u32)q;  // d wraps only on a cycle without separator, which is rejected
        mv = (u32)q != s;
    }
    if (__any_sync(0xffffffffu, mv) && lane_id() == 0) atomicExch(moved, 1u);
}
// requested string i: len_i = d[i], owner[succ[i]] = i
static __global__ void __launch_bounds__(INV_THREADS) inv_jump_owner_kernel(const u64* __restrict__ P, u32 n_req, u32* __restrict__ len, u32* __restrict__ owner) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_req) return;
    const u64 p = P[i];
    len[i] = (u32)(p >> 32);
    owner[(u32)p] = i;
}
// every non-separator row j stores BWT[j] at off[owner[succ[j]]] + d[j] - 1; a row whose chain ends on a row that is not a
// separator row lies on a cycle without separator (*bad); each requested string's last cell is its separator
template <class CellT>
__global__ void __launch_bounds__(INV_THREADS) inv_jump_scatter_kernel(const u64* __restrict__ E, const u64* __restrict__ P, const u32* __restrict__ owner, const u32* __restrict__ off,
                                                                       const u32* __restrict__ len, u32 n, u32 n_req, u32 sep, CellT* __restrict__ out, u32* bad) {
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    if (j < n_req) out[(u64)off[j] + j + len[j]] = (CellT)sep;  // string i starts at off[i] + i
    const u64 e = E[j];
    if (inv_sym(e) == sep) return;
    const u64 p = P[j];
    const u32 s = ld_gather4(owner + (u32)p);
    if (s == INV_NOT_SEP) { atomicExch(bad, 1u); return; }
    if (s == INV_UNREQ) return;
    out[(u64)ld_gather4(off + s) + s + (u32)(p >> 32) - 1] = (CellT)inv_sym(e);
}


template <class CellT>
void inv_walk_write(const u64* E, u32 n_req, u32 sep, const u32* len, const u32* off, u8* out, cudaStream_t st, u64 n_out) {
    GRL_LAUNCH("inv_walk_write", 2 * (n_out - n_req) * 32 + n_out * sizeof(CellT), (inv_walk_write_kernel<CellT>), grid_for(n_req, INV_THREADS), INV_THREADS, 0, st, E, n_req, sep, len,
               off, out);
}
template <class CellT>
void inv_jump_scatter(const u64* E, const u64* P, const u32* owner, const u32* off, const u32* len, u32 n, u32 n_req, u32 sep, u8* out, u32* bad, cudaStream_t st) {
    GRL_LAUNCH("inv_jump_scatter", (u64)n * (8 + 8 + 32 + 32 + 32), (inv_jump_scatter_kernel<CellT>), grid_for(n, INV_THREADS), INV_THREADS, 0, st, E, P, owner, off, len, n, n_req,
               sep, (CellT*)out, bad);
}

// pointer jumping to convergence (part c, shared with the locate table of fm.cuh): P[j] = {steps from j to its separator row << 32 |
// that row}; owner[] as inv_jump_init leaves it. Returns the rounds; GRLGPU_ERR_ILL_FORMED when it does not converge (the message
// starts with `who`, the caller's name for itself).
inline u32 inv_jump_converge(const u64* E, u32 n, u32 sep, DevBuf<u64>& P, u32* owner, u32* flag, cudaStream_t st, const char* who) {
    GRL_LAUNCH("inv_jump_init", (u64)n * 20, inv_jump_init_kernel, grid_for(n, INV_THREADS), INV_THREADS, 0, st, E, n, sep, P.p, owner);
    DevBuf<u64> Q(n, st);
    // after k rounds succ = LF^(2^k) stopped at the separator row, so ceil(log2 n) rounds converge any BWT and one more
    // moves nothing; an entry still moving after that lies on a cycle without separator
    const u32 cap = (u32)bit_width64(n - 1) + 1;
    bool moved = true;
    u32 rounds = 0;
    while (moved && rounds < cap) {  // at most cap rounds
        GRL_CUDA(cudaMemsetAsync(flag, 0, 4, st));
        GRL_LAUNCH("inv_jump_round", (u64)n * (8 + 32 + 8), inv_jump_round_kernel, grid_for(n, INV_THREADS), INV_THREADS, 0, st, P.p, n, Q.p, flag);
        std::swap(P, Q);
        rounds++;
        moved = d2h_scalar(flag, st) != 0;
    }
    if (moved) throw Error(GRLGPU_ERR_ILL_FORMED, std::string(who) + ": pointer jumping did not converge (an LF cycle without separator)");
    return rounds;
}

// the walk's step bound B = max(INV_B_MIN, n / INV_B_DIV), at most n: the inversion's count pass and fm.cuh's locate walk
inline u64 inv_walk_bound(u64 n) { return std::min<u64>(n, std::max<u64>(INV_B_MIN, n / INV_B_DIV)); }

// Part a on a checked image ([sb][fb] in 1..8, a whole number of records, at least one): decode, run starts, F rows, LF table,
// into `t`. The inversion needs only E and frees the rest; the FM-index (fm.cuh) keeps it all. With `sorted_keys` the symbol-sorted
// run order stays in t.order and the sorted symbols are handed over for the index's symbol directory (only when n > 0). Error
// messages start with `who`, the caller's name for itself.
inline void lf_table_build(const u8* image, u64 image_bytes, LfTable& t, DevBuf<u32>* sorted_keys, cudaStream_t st, const char* who) {
    const u64 sb = ((const u64*)image)[0], fb = ((const u64*)image)[1], rec = sb + fb, nr = (image_bytes - 16) / rec;
    t.n_runs = nr;
    t.sym.alloc(nr, st);
    t.len.alloc(nr, st);
    u32 h[3];  // does not fit 32 bits, largest symbol, separator
    {
        DevBuf<u8> raw(nr * rec, st);
        DevBuf<u32> stv(3, st);
        const u32 init[3] = {0u, 0u, 0xffffffffu};
        GRL_CUDA(cudaMemcpyAsync(raw.p, image + 16, nr * rec, cudaMemcpyHostToDevice, st));
        GRL_CUDA(cudaMemcpyAsync(stv.p, init, sizeof(init), cudaMemcpyHostToDevice, st));
        GRL_LAUNCH("inv_decode", nr * (rec + 8), inv_decode_kernel, grid_for(nr, INV_THREADS), INV_THREADS, 0, st, raw.p, nr, (int)sb, (int)fb, t.sym.p, t.len.p, stv.p);
        d2h_small(h, stv.p, sizeof(h), st);  // synchronises the stream: `init` is no longer read
    }
    if (h[0]) throw Error(GRLGPU_ERR_LIMIT, std::string(who) + ": a symbol or a run length of the image does not fit 32 bits");
    u64 n = 0;
    {
        DevBuf<u64> start64(nr, st), tot(1, st);
        exclusive_scan<u32, u64>(t.len.p, start64.p, nr, tot.p, st);
        n = d2h_scalar(tot.p, st);
    }
    if (n >= 0xfffffff0ull) throw Error(GRLGPU_ERR_LIMIT, std::string(who) + ": the BWT has 2^32 symbols or more");
    t.n = n;
    t.sep = h[2];
    t.E.alloc(n, st);
    t.N = 0;
    if (!n) return;
    {
        DevBuf<u64> cnt(1, st);
        cnt.zero();
        GRL_LAUNCH("inv_sep_count", nr * 8, inv_sep_count_kernel, grid_for(nr, INV_THREADS), INV_THREADS, 0, st, t.sym.p, t.len.p, nr, t.sep, cnt.p);
        t.N = d2h_scalar(cnt.p, st);
    }
    t.start.alloc(nr + 1, st);
    t.F.alloc(nr, st);
    exclusive_scan<u32, u32>(t.len.p, t.start.p, nr, t.start.p + nr, st);
    {   // stable sort of the run indices by symbol, lengths scanned in that order, scattered back to the runs
        DevBuf<u32> keys(nr, st), keys_alt(nr, st), vals(nr, st), vals_alt(nr, st);
        GRL_CUDA(cudaMemcpyAsync(keys.p, t.sym.p, nr * 4, cudaMemcpyDeviceToDevice, st));
        GRL_LAUNCH("inv_iota", nr * 4, inv_iota_kernel, grid_for(nr, INV_THREADS), INV_THREADS, 0, st, vals.p, nr);
        u32 *kp = keys.p, *vp = vals.p, *ka = keys_alt.p, *va = vals_alt.p;
        radix_sort_pairs_u32(&kp, &vp, &ka, &va, nr, std::max(1, bit_width64(h[1])), st);
        u32* fpos = ka;  // the alternate key buffer is free after the sort
        GRL_LAUNCH("inv_sorted_len", nr * 12, inv_sorted_len_kernel, grid_for(nr, INV_THREADS), INV_THREADS, 0, st, vp, t.len.p, nr, fpos);
        exclusive_scan<u32, u32>(fpos, fpos, nr, (u32*)nullptr, st);
        GRL_LAUNCH("inv_scatter_f", nr * 12, inv_scatter_f_kernel, grid_for(nr, INV_THREADS), INV_THREADS, 0, st, vp, fpos, nr, t.F.p);
        GRL_CUDA(cudaStreamSynchronize(st));
        if (sorted_keys) {  // the buffers that hold the sorted symbols and the order after the sort
            *sorted_keys = std::move(kp == keys.p ? keys : keys_alt);
            t.order = std::move(vp == vals.p ? vals : vals_alt);
        }
    }
    GRL_LAUNCH("inv_fill", n * 8 + nr * 12, inv_fill_kernel, (unsigned)div_up(n, INV_FILL_TILE), INV_THREADS, 0, st, t.start.p, t.F.p, t.sym.p, (u32)nr, (u32)n, t.E.p);
    GRL_CUDA(cudaStreamSynchronize(st));
}

// The whole inversion of a checked image (as lf_table_build): fills *info, and `out` when n_out * w <= cap_bytes
// (GRLGPU_ERR_ARG otherwise, with info->n_out set). Every buffer comes from the context's pool.
inline void invert_image(grlgpu_ctx* c, const u8* image, u64 image_bytes, int w, u64 n_seqs, void* out, u64 cap_bytes, grlgpu_invert_t* info) {
    cudaStream_t st = c->st;
    Timer t_all(st), t_lf(st), t_inv(st);
    t_all.start();
    t_lf.start();
    const u64 sb = ((const u64*)image)[0], fb = ((const u64*)image)[1];
    info->n_runs = (image_bytes - 16) / (sb + fb);
    // ---- a: decode, run starts, F positions, LF table ----
    LfTable t;
    lf_table_build(image, image_bytes, t, nullptr, st, "inversion on the device");
    info->n = t.n;
    t.start.release();
    t.F.release();
    t.sym.release();
    t.len.release();
    const u64 n = t.n, N = t.N;
    const u32 sep = t.sep;
    DevBuf<u64>& E = t.E;
    t_lf.stop();
    info->n_strings = N;
    const u32 n_req = (u32)std::min<u64>(n_seqs, N);
    // ---- b / c / d: inversion ----
    t_inv.start();
    DevBuf<u32> slen(n_req, st), off((u64)n_req + 1, st), flag(1, st);
    const bool force_walk = (c->flags & GRLGPU_FLAG_FORCE_WALK) != 0, force_jump = (c->flags & GRLGPU_FLAG_FORCE_JUMP) != 0 && !force_walk;
    bool walk = !force_jump;
    if (walk) {  // count pass: chains of rows < N end within n steps, so the bound n never overflows
        const u64 B = force_walk ? n : inv_walk_bound(n);
        flag.zero();
        GRL_LAUNCH("inv_walk_count", (u64)n_req * 4 + (n - N) * 32, inv_walk_count_kernel, grid_for(n_req, INV_THREADS), INV_THREADS, 0, st, E.p, (const u32*)nullptr, n_req, sep, (u32)B, slen.p, flag.p);
        walk = d2h_scalar(flag.p, st) == 0;
    }
    const auto sized = [&](u64 n_out) {  // output size known: check the caller's capacity
        info->n_out = n_out;
        if (n_out * (u64)w > cap_bytes) throw Error(GRLGPU_ERR_ARG, "inversion: the output needs " + std::to_string(n_out * (u64)w) + " bytes");
    };
    DevBuf<u8> dout;
    if (walk) {
        info->path = 0;
        exclusive_scan<u32, u32>(slen.p, off.p, n_req, off.p + n_req, st);
        const u64 n_out = (u64)d2h_scalar(off.p + n_req, st) + n_req;
        if (n_req == N && n_out != n) throw Error(GRLGPU_ERR_ILL_FORMED, "inversion: the strings do not cover the BWT (an LF cycle without separator)");
        sized(n_out);
        dout.alloc(n_out * w + 16, st);
        switch (w) {
            case 1: inv_walk_write<u8>(E.p, n_req, sep, slen.p, off.p, dout.p, st, n_out); break;
            case 2: inv_walk_write<u16>(E.p, n_req, sep, slen.p, off.p, dout.p, st, n_out); break;
            case 4: inv_walk_write<u32>(E.p, n_req, sep, slen.p, off.p, dout.p, st, n_out); break;
            default: inv_walk_write<u64>(E.p, n_req, sep, slen.p, off.p, dout.p, st, n_out); break;
        }
    } else {
        info->path = 1;
        DevBuf<u64> P(n, st);
        DevBuf<u32> owner(n, st);
        info->jump_rounds = inv_jump_converge(E.p, (u32)n, sep, P, owner.p, flag.p, st, "inversion");
        GRL_LAUNCH("inv_jump_owner", (u64)n_req * (8 + 4 + 32), inv_jump_owner_kernel, grid_for(n_req, INV_THREADS), INV_THREADS, 0, st, P.p, n_req, slen.p, owner.p);
        exclusive_scan<u32, u32>(slen.p, off.p, n_req, off.p + n_req, st);
        const u64 n_out = (u64)d2h_scalar(off.p + n_req, st) + n_req;
        sized(n_out);
        dout.alloc(n_out * w + 16, st);
        flag.zero();
        switch (w) {
            case 1: inv_jump_scatter<u8>(E.p, P.p, owner.p, off.p, slen.p, (u32)n, n_req, sep, dout.p, flag.p, st); break;
            case 2: inv_jump_scatter<u16>(E.p, P.p, owner.p, off.p, slen.p, (u32)n, n_req, sep, dout.p, flag.p, st); break;
            case 4: inv_jump_scatter<u32>(E.p, P.p, owner.p, off.p, slen.p, (u32)n, n_req, sep, dout.p, flag.p, st); break;
            default: inv_jump_scatter<u64>(E.p, P.p, owner.p, off.p, slen.p, (u32)n, n_req, sep, dout.p, flag.p, st); break;
        }
        if (d2h_scalar(flag.p, st)) throw Error(GRLGPU_ERR_ILL_FORMED, "inversion: a chain ends on a row that is not a separator row (an LF cycle without separator)");
    }
    t_inv.stop();
    if (info->n_out) GRL_CUDA(cudaMemcpyAsync(out, dout.p, info->n_out * (u64)w, cudaMemcpyDeviceToHost, st));
    t_all.stop();
    info->lf_ms = t_lf.ms();
    info->invert_ms = t_inv.ms();
    info->device_ms = t_all.ms();  // waits for the copy
}
