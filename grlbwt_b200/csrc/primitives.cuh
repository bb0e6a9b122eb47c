// Device-wide building blocks written for this path: exclusive scan, bitmap -> position compaction,
// LSD radix sort of (u64 or u32 key, u32 value) pairs and its one-digit partition, max-reduction.
// All are plain multi-kernel formulations (no inter-CTA spin waits), HBM-bound, grid sized from the data.
#pragma once
#include <type_traits>
#include "util.cuh"

namespace grl {

// ------------------------------------------------------------------------------------------------
// Exclusive scan: out[i] = op_{j<i} in[j]  (TOut accumulates; op is the sum unless Op says otherwise). Works in place (in == out).
// ------------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

// scan operators: associative, with identity 0 on the unsigned types they are used with
struct ScanSum {
    template <class T>
    __device__ __forceinline__ static T apply(T a, T b) { return a + b; }
};
struct ScanMax {
    template <class T>
    __device__ __forceinline__ static T apply(T a, T b) { return a > b ? a : b; }
};
template <class Op, class T>
__device__ __forceinline__ T warp_inclusive_op(T v) {
    const u32 l = lane_id();
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T x = __shfl_up_sync(0xffffffffu, v, o);
        if (l >= (u32)o) v = Op::apply(v, x);
    }
    return v;
}
// block_exclusive_sum (util.cuh) for any scan operator: the sum keeps its own code; other operators take the exclusive prefix of a
// lane from its neighbour's inclusive one, since they cannot subtract
template <class Op, class T>
__device__ __forceinline__ T block_exclusive_op(T v, T* smem, T& total) {
    if constexpr (std::is_same<Op, ScanSum>::value) {
        return block_exclusive_sum<T>(v, smem, total);
    } else {
        const u32 l = lane_id(), w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
        const T inc = warp_inclusive_op<Op>(v);
        T ex = __shfl_up_sync(0xffffffffu, inc, 1);
        if (l == 0) ex = T(0);
        if (l == 31) smem[w] = inc;
        __syncthreads();
        if (w == 0) {
            const T x = l < nw ? smem[l] : T(0);
            const T xi = warp_inclusive_op<Op>(x);
            T xe = __shfl_up_sync(0xffffffffu, xi, 1);
            if (l == 0) xe = T(0);
            smem[l] = xe;  // exclusive prefix of warp totals
            if (l == 31) smem[32] = xi;
        }
        __syncthreads();
        const T res = Op::apply(smem[w], ex);
        total = smem[32];
        __syncthreads();
        return res;
    }
}
// a thread's SCAN_ITEMS consecutive items move as 16-byte vectors when the whole run exists and the array is 16-byte aligned
template <class T>
__device__ __forceinline__ void scan_load(const T* in, u64 base, u64 n, bool vec, T (&v)[SCAN_ITEMS]) {
    constexpr int NV = SCAN_ITEMS * sizeof(T) / 16, PER = 16 / sizeof(T);
    if (vec && base + SCAN_ITEMS <= n) {
        const uint4* p = reinterpret_cast<const uint4*>(in + base);
#pragma unroll
        for (int q = 0; q < NV; q++) {
            const uint4 x = p[q];
            memcpy(&v[q * PER], &x, 16);
        }
    } else {
#pragma unroll
        for (int i = 0; i < SCAN_ITEMS; i++) v[i] = (base + i < n) ? in[base + i] : T(0);
    }
}
template <class T>
__device__ __forceinline__ void scan_store(T* out, u64 base, u64 n, bool vec, const T (&v)[SCAN_ITEMS]) {
    constexpr int NV = SCAN_ITEMS * sizeof(T) / 16, PER = 16 / sizeof(T);
    if (vec && base + SCAN_ITEMS <= n) {
        uint4* p = reinterpret_cast<uint4*>(out + base);
#pragma unroll
        for (int q = 0; q < NV; q++) {
            uint4 x;
            memcpy(&x, &v[q * PER], 16);
            p[q] = x;
        }
    } else {
#pragma unroll
        for (int i = 0; i < SCAN_ITEMS; i++)
            if (base + i < n) out[base + i] = v[i];
    }
}

template <class TIn, class TOut, class Op = ScanSum>
__global__ void __launch_bounds__(SCAN_THREADS) scan_tile_sums_kernel(const TIn* __restrict__ in, TOut* __restrict__ partial, u64 n, bool vec) {
    __shared__ TOut sm[33];
    const u64 base = (u64)blockIdx.x * SCAN_TILE + (u64)threadIdx.x * SCAN_ITEMS;
    TIn x[SCAN_ITEMS];
    scan_load<TIn>(in, base, n, vec, x);
    TOut s = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; i++) s = Op::apply(s, (TOut)x[i]);
    TOut tot;
    block_exclusive_op<Op, TOut>(s, sm, tot);
    if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}

// single block scans a short array (n <= any size, loops tile by tile), writes the grand total
template <class TIn, class TOut, class Op = ScanSum>
__global__ void __launch_bounds__(SCAN_THREADS) scan_single_block_kernel(const TIn* in, TOut* out, u64 n, TOut* total) {
    __shared__ TOut sm[33];
    TOut carry = 0;
    for (u64 t0 = 0; t0 < n; t0 += SCAN_TILE) {
        const u64 base = t0 + (u64)threadIdx.x * SCAN_ITEMS;
        TOut v[SCAN_ITEMS];
        TOut s = 0;
#pragma unroll
        for (int i = 0; i < SCAN_ITEMS; i++) {
            v[i] = (base + i < n) ? (TOut)in[base + i] : TOut(0);
            s = Op::apply(s, v[i]);
        }
        TOut tot;
        TOut ex = Op::apply(block_exclusive_op<Op, TOut>(s, sm, tot), carry);
#pragma unroll
        for (int i = 0; i < SCAN_ITEMS; i++) {
            if (base + i < n) out[base + i] = ex;
            ex = Op::apply(ex, v[i]);
        }
        carry = Op::apply(carry, tot);
    }
    if (threadIdx.x == 0 && total) *total = carry;
}

template <class TIn, class TOut, class Op = ScanSum>
__global__ void __launch_bounds__(SCAN_THREADS) scan_apply_kernel(const TIn* in, TOut* out, const TOut* __restrict__ tile_prefix, u64 n, bool vec) {
    __shared__ TOut sm[33];
    const u64 base = (u64)blockIdx.x * SCAN_TILE + (u64)threadIdx.x * SCAN_ITEMS;
    TIn x[SCAN_ITEMS];
    scan_load<TIn>(in, base, n, vec, x);
    TOut s = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; i++) s = Op::apply(s, (TOut)x[i]);
    TOut tot;
    TOut ex = Op::apply(block_exclusive_op<Op, TOut>(s, sm, tot), tile_prefix[blockIdx.x]);
    TOut v[SCAN_ITEMS];
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; i++) {
        v[i] = ex;
        ex = Op::apply(ex, (TOut)x[i]);
    }
    scan_store<TOut>(out, base, n, vec, v);
}

// total_dev (optional, device pointer) receives the op of all inputs (the sum, or with ScanMax the maximum).
template <class TIn, class TOut, class Op = ScanSum>
void exclusive_scan(const TIn* in, TOut* out, u64 n, TOut* total_dev, cudaStream_t st) {
    if (n <= (u64)SCAN_TILE * 4) {
        GRL_LAUNCH("scan_single_block", n * (sizeof(TIn) + sizeof(TOut)), (scan_single_block_kernel<TIn, TOut, Op>), 1, SCAN_THREADS, 0, st, in, out, n, total_dev);
        return;
    }
    const u64 tiles = div_up(n, SCAN_TILE);
    DevBuf<TOut> partial(tiles, st);
    const bool vec = (((uintptr_t)in | (uintptr_t)out) & 15) == 0;
    GRL_LAUNCH("scan_tile_sums", n * sizeof(TIn), (scan_tile_sums_kernel<TIn, TOut, Op>), (unsigned)tiles, SCAN_THREADS, 0, st, in, partial.p, n, vec);
    exclusive_scan<TOut, TOut, Op>(partial.p, partial.p, tiles, total_dev, st);
    GRL_LAUNCH("scan_apply", n * (sizeof(TIn) + sizeof(TOut)), (scan_apply_kernel<TIn, TOut, Op>), (unsigned)tiles, SCAN_THREADS, 0, st, in, out, partial.p, n, vec);
}

// ------------------------------------------------------------------------------------------------
// Bitmap compaction: positions of the set bits of `bits` (n_bits bits, u32 words, LSB first), in
// increasing order. If `prev_bits` is given, the output carries a flag in its top bit:
// flag(q) = (q == 0) || prev_bits[q-1]   (used as "q starts a string" when prev_bits marks string ends).
// ------------------------------------------------------------------------------------------------
constexpr int BC_THREADS = 256;
constexpr int BC_WORDS = 8;                      // words per thread
constexpr int BC_TILE_WORDS = BC_THREADS * BC_WORDS;

__device__ __forceinline__ u32 bc_load_word(const u32* __restrict__ bits, u64 w, u64 n_words, u64 n_bits) {
    if (w >= n_words) return 0;
    u32 x = bits[w];
    if (w == n_words - 1 && (n_bits & 31)) x &= (1u << (n_bits & 31)) - 1u;
    return x;
}

static __global__ void __launch_bounds__(BC_THREADS) bitmap_count_kernel(const u32* __restrict__ bits, u64 n_bits, u32* __restrict__ tile_count) {
    __shared__ u32 sm[33];
    const u64 n_words = (n_bits + 31) / 32;
    const u64 w0 = (u64)blockIdx.x * BC_TILE_WORDS + (u64)threadIdx.x * BC_WORDS;
    u32 c = 0;
#pragma unroll
    for (int i = 0; i < BC_WORDS; i++) c += __popc(bc_load_word(bits, w0 + i, n_words, n_bits));
    u32 tot;
    block_exclusive_sum<u32>(c, sm, tot);
    if (threadIdx.x == 0) tile_count[blockIdx.x] = tot;
}

// A warp owns 32 * BC_WORDS consecutive words and walks them 32 at a time (lane = word): the positions of one step go
// through a 1024-entry shared-memory stage (10-bit offset | flag << 15) so that the stores to `out` are coalesced.
template <class PosT>
__global__ void __launch_bounds__(BC_THREADS) bitmap_write_kernel(const u32* __restrict__ bits, const u32* __restrict__ prev_bits, u64 n_bits,
                                                                  const u64* __restrict__ tile_off, PosT* __restrict__ out) {
    __shared__ u32 wtot[BC_THREADS / 32];
    __shared__ unsigned short stage[BC_THREADS / 32][1024];
    constexpr PosT FLAG = PosT(1) << (sizeof(PosT) * 8 - 1);
    const u32 lane = lane_id(), warp = threadIdx.x >> 5;
    const u64 n_words = (n_bits + 31) / 32;
    const u64 wbase = (u64)blockIdx.x * BC_TILE_WORDS + (u64)warp * (32 * BC_WORDS);
    u32 wd[BC_WORDS];
    u32 c = 0;
#pragma unroll
    for (int i = 0; i < BC_WORDS; i++) {
        wd[i] = bc_load_word(bits, wbase + (u64)i * 32 + lane, n_words, n_bits);
        c += __popc(wd[i]);
    }
    c = warp_sum(c);
    if (lane == 0) wtot[warp] = c;
    __syncthreads();
    u64 o = tile_off[blockIdx.x];
    for (u32 w2 = 0; w2 < warp; w2++) o += wtot[w2];
#pragma unroll
    for (int i = 0; i < BC_WORDS; i++) {
        u32 x = wd[i];
        const u32 cnt = __popc(x);
        const u32 inc = warp_inclusive_sum(cnt);
        const u32 T = __shfl_sync(0xffffffffu, inc, 31);
        if (T == 0) continue;
        u32 ex = inc - cnt;
        u32 fl = 0;
        if (prev_bits && x) {
            const u64 w = wbase + (u64)i * 32 + lane;
            const u32 pw = bc_load_word(prev_bits, w, n_words, n_bits);
            const u32 pp = w ? bc_load_word(prev_bits, w - 1, n_words, n_bits) : 0x80000000u;  // position 0 starts a string
            fl = (pw << 1) | (pp >> 31);
        }
        while (x) {
            const int b = __ffs(x) - 1;
            x &= x - 1;
            stage[warp][ex++] = (unsigned short)((lane << 5) | (u32)b | (((fl >> b) & 1u) << 15));
        }
        __syncwarp();
        const u64 bit_base = (wbase + (u64)i * 32) * 32;
        for (u32 j = lane; j < T; j += 32) {
            const u32 sv = stage[warp][j];
            PosT q = (PosT)(bit_base + (sv & 0x3ffu));
            if (sv >> 15) q |= FLAG;
            out[o + j] = q;
        }
        __syncwarp();
        o += T;
    }
}

// Returns the number of set bits (host value; synchronises the stream). out must hold count entries:
// call with out == nullptr first to size it, or give an upper bound. Here: two-phase API.
struct BitmapCompactor {
    DevBuf<u32> tile_count;
    DevBuf<u64> tile_off;
    DevBuf<u64> total;
    u64 n_bits = 0, tiles = 0;
    const u32* bits = nullptr;
    cudaStream_t st = nullptr;
    // phase 1: count
    u64 count(const u32* bits_, u64 n_bits_, cudaStream_t s) {
        bits = bits_; n_bits = n_bits_; st = s;
        const u64 n_words = (n_bits + 31) / 32;
        tiles = div_up(n_words ? n_words : 1, BC_TILE_WORDS);
        tile_count.alloc(tiles, st);
        tile_off.alloc(tiles, st);
        total.alloc(1, st);
        GRL_LAUNCH("bitmap_count", n_bits / 8, bitmap_count_kernel, (unsigned)tiles, BC_THREADS, 0, st, bits, n_bits, tile_count.p);
        exclusive_scan<u32, u64>(tile_count.p, tile_off.p, tiles, total.p, st);
        u64 h = 0;
        d2h_small(&h, total.p, sizeof(u64), st);
        return h;
    }
    // phase 2: write positions
    template <class PosT>
    void write(const u32* prev_bits, PosT* out) {
        GRL_LAUNCH("bitmap_write", n_bits / 4, (bitmap_write_kernel<PosT>), (unsigned)tiles, BC_THREADS, 0, st, bits, prev_bits, n_bits, tile_off.p, out);
    }
};

// ------------------------------------------------------------------------------------------------
// LSD radix sort of (u64 or u32 key, u32 value) pairs on key bits [0, n_bits), 8 bits per pass, stable. n_bits is rounded up
// to whole 8-bit digits; key bits above those are carried unsorted.
// Per pass: per-tile digit histogram -> exclusive scan of the digit-major table -> ranked scatter
// through shared memory (writes of one digit from one tile are contiguous).
// ------------------------------------------------------------------------------------------------
constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_ITEMS = 8;  // items per thread: 59 registers, 4 CTAs/SM (measured best on B200 against 4, 12 and 16)
template <class KeyT, int ITEMS>
constexpr size_t rs_smem_bytes() {
    return (size_t)RS_THREADS * ITEMS * (sizeof(KeyT) + sizeof(u32)) + (size_t)RS_WARPS * 257 * sizeof(u32) + 2 * 256 * sizeof(u32) + 34 * sizeof(u32);
}

template <class KeyT, int ITEMS>
__global__ void __launch_bounds__(RS_THREADS) radix_hist_kernel(const KeyT* __restrict__ keys, u64 n, int shift, u32* __restrict__ hist, u64 tiles) {
    __shared__ u32 cnt[256];
    cnt[threadIdx.x] = 0;
    const u64 base = (u64)blockIdx.x * (RS_THREADS * ITEMS);
    KeyT k[ITEMS];
#pragma unroll
    for (int i = 0; i < ITEMS; i++) {  // all loads in flight before the first atomic
        const u64 idx = base + (u64)i * RS_THREADS + threadIdx.x;
        k[i] = idx < n ? keys[idx] : (KeyT)0;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < ITEMS; i++) {
        const u64 idx = base + (u64)i * RS_THREADS + threadIdx.x;
        if (idx < n) atomicAdd(&cnt[(u32)(k[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[(u64)threadIdx.x * tiles + blockIdx.x] = cnt[threadIdx.x];
}

template <class KeyT, int ITEMS>
__global__ void __launch_bounds__(RS_THREADS, 4) radix_scatter_kernel(const KeyT* __restrict__ keys_in, const u32* __restrict__ vals_in, KeyT* __restrict__ keys_out,
                                                                   u32* __restrict__ vals_out, u64 n, int shift, const u64* __restrict__ goff, u64 tiles) {
    constexpr int TILE = RS_THREADS * ITEMS, WARP_ITEMS = TILE / RS_WARPS;
    extern __shared__ __align__(16) unsigned char rs_smem[];
    KeyT* s_keys = (KeyT*)rs_smem;
    u32* s_vals = (u32*)(s_keys + TILE);
    u32* s_cnt = s_vals + TILE;               // [RS_WARPS][257]
    u32* s_dstart = s_cnt + RS_WARPS * 257;   // [256] tile-local start of each digit
    u32* s_scan = s_dstart + 256;             // 33 scratch
    __shared__ u64 s_delta[256];              // global offset of digit d minus its tile-local start

    const u32 lane = lane_id(), warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < RS_WARPS * 257; i += RS_THREADS) s_cnt[i] = 0;
    __syncthreads();

    const u64 tile_base = (u64)blockIdx.x * TILE;
    KeyT key[ITEMS];
    u32 val[ITEMS];
    u32 rnk[ITEMS];
    u32* wc = s_cnt + warp * 257;
#pragma unroll
    for (int r = 0; r < ITEMS; r++) {
        const u64 idx = tile_base + (u64)warp * WARP_ITEMS + (u64)r * 32 + lane;
        const bool ok = idx < n;
        key[r] = ok ? keys_in[idx] : (KeyT)~(KeyT)0;
        val[r] = ok ? vals_in[idx] : 0u;
        const u32 d = ok ? ((u32)(key[r] >> shift) & 255u) : 256u;
        const u32 m = __match_any_sync(0xffffffffu, d);
        const u32 b = wc[d];
        __syncwarp();
        if (lane == (u32)(__ffs(m) - 1)) wc[d] = b + __popc(m);
        __syncwarp();
        rnk[r] = b + __popc(m & lanemask_lt());
    }
    __syncthreads();
    // per digit: exclusive prefix over warps, tile count
    {
        const u32 d = threadIdx.x;
        const u64 my_goff = goff[(u64)d * tiles + blockIdx.x];
        u32 c[RS_WARPS], run = 0;
#pragma unroll
        for (int w = 0; w < RS_WARPS; w++) { c[w] = s_cnt[w * 257 + d]; run += c[w]; }
        u32 tot;
        u32 ex = block_exclusive_sum<u32>(run, s_scan, tot);
        s_delta[d] = my_goff - ex;
#pragma unroll
        for (int w = 0; w < RS_WARPS; w++) { s_cnt[w * 257 + d] = ex; ex += c[w]; }  // tile-local start of (warp, digit)
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < ITEMS; r++) {
        const u64 idx = tile_base + (u64)warp * WARP_ITEMS + (u64)r * 32 + lane;
        if (idx < n) {
            const u32 d = (u32)(key[r] >> shift) & 255u;
            const u32 pos = wc[d] + rnk[r];
            s_keys[pos] = key[r];
            s_vals[pos] = val[r];
        }
    }
    __syncthreads();
    const u64 rem = n - tile_base;
    const u32 valid = rem < (u64)TILE ? (u32)rem : (u32)TILE;
    for (u32 i = threadIdx.x; i < valid; i += RS_THREADS) {
        const KeyT k = s_keys[i];
        const u32 d = (u32)(k >> shift) & 255u;
        const u64 g = s_delta[d] + i;
        keys_out[g] = k;
        vals_out[g] = s_vals[i];
    }
}

// one stable partition pass on the 8-bit digit at `shift` (also the building block of the LSD sort below)
template <class KeyT>
inline void radix_pass(KeyT** keys, u32** vals, KeyT** keys_alt, u32** vals_alt, u64 n, int shift, DevBuf<u32>& hist, DevBuf<u64>& goff, cudaStream_t st) {
    // per-device attribute: (re)applied for the current device, not cached process-wide
    GRL_CUDA(cudaFuncSetAttribute(radix_scatter_kernel<KeyT, RS_ITEMS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rs_smem_bytes<KeyT, RS_ITEMS>()));
    const u64 tiles = div_up(n, RS_THREADS * RS_ITEMS);
    GRL_LAUNCH("radix_hist", n * sizeof(KeyT), (radix_hist_kernel<KeyT, RS_ITEMS>), (unsigned)tiles, RS_THREADS, 0, st, *keys, n, shift, hist.p, tiles);
    exclusive_scan<u32, u64>(hist.p, goff.p, 256 * tiles, nullptr, st);
    GRL_LAUNCH("radix_scatter", n * 2 * (sizeof(KeyT) + 4), (radix_scatter_kernel<KeyT, RS_ITEMS>), (unsigned)tiles, RS_THREADS, (rs_smem_bytes<KeyT, RS_ITEMS>()), st, *keys,
               *vals, *keys_alt, *vals_alt, n, shift, goff.p, tiles);
    KeyT* tk = *keys; *keys = *keys_alt; *keys_alt = tk;
    u32* tv = *vals; *vals = *vals_alt; *vals_alt = tv;
}
// Sorts in place logically: on return *keys / *vals point at the buffers holding the sorted data
// (either the inputs or the alternates).
inline void radix_sort_pairs(u64** keys, u32** vals, u64** keys_alt, u32** vals_alt, u64 n, int n_bits, cudaStream_t st) {
    if (n <= 1 || n_bits <= 0) return;
    const u64 tiles = div_up(n, RS_THREADS * RS_ITEMS);
    DevBuf<u32> hist(256 * tiles, st);
    DevBuf<u64> goff(256 * tiles, st);
    for (int shift = 0; shift < n_bits; shift += 8) radix_pass<u64>(keys, vals, keys_alt, vals_alt, n, shift, hist, goff, st);
}
// (u32 key, u32 value) pairs partitioned by the key's digit at `shift`: used to make a big random scatter L2-local
inline void radix_partition_u32(u32** keys, u32** vals, u32** keys_alt, u32** vals_alt, u64 n, int shift, cudaStream_t st) {
    const u64 tiles = div_up(n, RS_THREADS * RS_ITEMS);
    DevBuf<u32> hist(256 * tiles, st);
    DevBuf<u64> goff(256 * tiles, st);
    radix_pass<u32>(keys, vals, keys_alt, vals_alt, n, shift, hist, goff, st);
}
// LSD sort of (u32 key, u32 value) pairs on the low n_bits of the key
inline void radix_sort_pairs_u32(u32** keys, u32** vals, u32** keys_alt, u32** vals_alt, u64 n, int n_bits, cudaStream_t st) {
    if (n <= 1 || n_bits <= 0) return;
    const u64 tiles = div_up(n, RS_THREADS * RS_ITEMS);
    DevBuf<u32> hist(256 * tiles, st);
    DevBuf<u64> goff(256 * tiles, st);
    for (int shift = 0; shift < n_bits; shift += 8) radix_pass<u32>(keys, vals, keys_alt, vals_alt, n, shift, hist, goff, st);
}

// ------------------------------------------------------------------------------------------------
// max-reduction of a u64 array into *out (device, must be zeroed by the caller)
// ------------------------------------------------------------------------------------------------
static __global__ void reduce_max_u64_kernel(const u64* __restrict__ in, u64 n, u64* out) {
    u64 m = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) m = in[i] > m ? in[i] : m;
    m = warp_max(m);
    if (lane_id() == 0 && m) atomicMax(out, m);
}

}  // namespace grl
