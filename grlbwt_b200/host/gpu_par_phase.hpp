// Host side of the parse phase: drives the device library (include/grlgpu.h) round by round and collects what the
// induction phase needs. Replaces exact_algo::par_phase<sym_type> (lib/exact_algo/exact_par_phase.cpp:285-372) and, for
// several GPUs, the thread fan-out of mt_parse_strat_t (include/parsing_strategies.h:244-275): one host thread per GPU,
// each owning a shard of whole strings, exchanging through NCCL or peer copies inside the device library.
//
// I/O pipeline (SURVEY.md 8(f)-3): the input streams from the file (or from memory) through two pinned staging buffers,
// so reading chunk k+1 overlaps the host-to-device copy of chunk k (the reference reads 8 MB windows,
// external/cdt/include/file_streams.hpp:93-105); every level's artefacts are handed to fetch threads that copy them to
// the host while the device computes the next round (the reference writes dict_lev_k / pre_bwt_lev_k files between
// rounds, exact_par_phase.cpp:150-155,:402-406).
#pragma once
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <array>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <iostream>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/grlgpu.h"
#include "ind_phase.hpp"
#include "ind_phase_mt.hpp"

namespace grlbwt {

struct GpuError : std::runtime_error {
    int status;
    GpuError(int st, const std::string& m) : std::runtime_error(m), status(st) {}
};

inline double ms_since(std::chrono::steady_clock::time_point t0) {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

// what one round left behind, for parity checks across GPU counts: the level's global sizes and four order-insensitive sums
// over its rules / hocc marks / preliminary BWT (grlgpu_level_checksum; the slices of a multi-GPU level add up to the same)
struct RoundDigest {
    uint64_t tot = 0, n_pre = 0, parse_len = 0, n_phrases = 0, dict_syms = 0;
    uint64_t cs[4] = {0, 0, 0, 0};
};

struct ParseResult {
    grlgpu_stats_t stats{};
    std::vector<Level> levels;        // 64-bit symbols: only filled when some level needs them
    std::vector<Level32> levels32;    // 32-bit symbols (the usual case), consumed by the multi-threaded induction
    bool wide = false;
    std::vector<grlgpu_round_t> rounds;
    std::vector<RoundDigest> digests;
    std::vector<uint64_t> final_parse;  // one cell per string, cells = rank<<1|rep
    double h2d_ms = 0, par_ms = 0;
    uint64_t exchange_bytes = 0;        // multi-GPU: bulk bytes sent between the ranks, all rounds, all ranks
    int n_ranks = 1;
    std::string comm_kind;
    // induction on the device (include/grlgpu.h: grlgpu_keep_level / grlgpu_induce): the level-0 BWT, levels stay empty
    bool induced_on_device = false;
    double dev_ind_ms = 0, dev_ind_compute_ms = 0;
    RunArr bwt_dev;
    uint64_t packed_bytes = 0;           // size of the .rl_bwt image written to OutputBuffers::packed
    bool bwt_in_caller_buffers = false;  // the runs were written to the caller's OutputBuffers (bwt_dev holds only the count)
};

// caller-owned landing zone for the level-0 BWT of the device induction (32-bit symbols and lengths); pinned memory makes the
// copy-back a plain DMA instead of a first-touch of fresh pages
struct OutputBuffers {
    uint32_t* sym = nullptr;
    uint32_t* len = nullptr;
    uint64_t cap = 0;  // runs each array can hold
    // alternatively: the image of the .rl_bwt file ([sb][fb] + records of sb + fb bytes), packed on the device
    unsigned char* packed = nullptr;
    uint64_t packed_cap = 0;  // bytes
};

// the input of the parse phase: a buffer in host memory or a byte range of a file
struct TextSource {
    const unsigned char* mem = nullptr;
    std::string file;
    uint64_t offset = 0, bytes = 0;
};

// ---------------------------------------------------------------- fetch threads
class FetchPool {
    struct Job { int device; void* dst; const void* src; uint64_t bytes; };
    std::vector<std::thread> th;
    std::mutex m;
    std::condition_variable cv, cv_done;
    std::deque<Job> q;
    size_t pending = 0;
    bool stop = false;
    int err = 0;
    void work() {
        for (;;) {
            Job j;
            {
                std::unique_lock<std::mutex> lk(m);
                cv.wait(lk, [&] { return stop || !q.empty(); });
                if (q.empty()) return;
                j = q.front();
                q.pop_front();
            }
            // large arrays are cut into pieces so that several threads share one array's copy
            const int rc = grlgpu_copy_to_host(j.device, j.dst, j.src, j.bytes);
            std::lock_guard<std::mutex> lk(m);
            if (rc != GRLGPU_OK && !err) err = rc;
            if (--pending == 0) cv_done.notify_all();
        }
    }

public:
    explicit FetchPool(size_t n_threads) {
        for (size_t t = 0; t < std::max<size_t>(1, n_threads); t++) th.emplace_back([this] { work(); });
    }
    ~FetchPool() {
        { std::lock_guard<std::mutex> lk(m); stop = true; }
        cv.notify_all();
        for (auto& t : th) t.join();
    }
    void enqueue(int device, void* dst, const void* src, uint64_t bytes) {
        constexpr uint64_t PIECE = 256ull << 20;
        std::lock_guard<std::mutex> lk(m);
        for (uint64_t o = 0; o < bytes; o += PIECE) {
            q.push_back({device, (char*)dst + o, (const char*)src + o, std::min(PIECE, bytes - o)});
            pending++;
        }
        cv.notify_all();
    }
    void wait_all() {
        std::unique_lock<std::mutex> lk(m);
        cv_done.wait(lk, [&] { return pending == 0; });
        if (err) { const int e = err; err = 0; throw GpuError(e, std::string("level fetch: ") + grlgpu_strerror(e)); }
    }
};

// ---------------------------------------------------------------- small helpers
struct CtxHandle {  // RAII around grlgpu_ctx
    grlgpu_ctx* p = nullptr;
    CtxHandle(int device, uint64_t flags) {
        const int rc = grlgpu_create(&p, device, flags);
        if (rc != GRLGPU_OK) throw GpuError(rc, std::string("grlgpu_create: ") + grlgpu_strerror(rc));
    }
    CtxHandle(const CtxHandle&) = delete;
    ~CtxHandle() { if (p) grlgpu_destroy(p); }
    void check(const char* what, int st) const {
        if (st != GRLGPU_OK) throw GpuError(st, std::string(what) + ": " + grlgpu_strerror(st) + " (" + grlgpu_last_error(p) + ")");
    }
};

// text -> device through the pinned staging buffers; returns the milliseconds it took
inline double load_text(const CtxHandle& ctx, const TextSource& src, int sym_bytes) {
    const auto t0 = std::chrono::steady_clock::now();
    if (src.bytes == 0 || src.bytes % (uint64_t)sym_bytes) throw GpuError(GRLGPU_ERR_ILL_FORMED, "the input is empty or not a whole number of symbols");
    if (src.mem) {  // already in host memory: one copy call (the driver stages pageable memory at ~10 GB/s; a caller with pinned memory gets DMA rate)
        ctx.check("grlgpu_set_text", grlgpu_set_text(ctx.p, src.mem + src.offset, src.bytes / (uint64_t)sym_bytes, sym_bytes));
        return ms_since(t0);
    }
    ctx.check("grlgpu_text_begin", grlgpu_text_begin(ctx.p, src.bytes / (uint64_t)sym_bytes, sym_bytes, 0));
    const int fd = open(src.file.c_str(), O_RDONLY);
    if (fd < 0) throw std::runtime_error("cannot open " + src.file);
    posix_fadvise(fd, (off_t)src.offset, (off_t)src.bytes, POSIX_FADV_SEQUENTIAL);
    try {
        for (uint64_t done = 0; done < src.bytes;) {
            void* buf = nullptr;
            uint64_t cap = 0;
            ctx.check("grlgpu_text_stage", grlgpu_text_stage(ctx.p, &buf, &cap));
            uint64_t got = 0;
            while (got < cap) {
                const ssize_t r = pread(fd, (char*)buf + got, cap - got, (off_t)(src.offset + done + got));
                if (r <= 0) throw std::runtime_error("cannot read " + src.file);
                got += (uint64_t)r;
            }
            ctx.check("grlgpu_text_commit", grlgpu_text_commit(ctx.p, got));
            done += got;
        }
        ctx.check("grlgpu_text_end", grlgpu_text_end(ctx.p));
    } catch (...) {
        close(fd);
        throw;
    }
    close(fd);
    return ms_since(t0);
}

inline uint64_t read_cell(const TextSource& src, int fd, uint64_t cell, int w) {
    uint64_t v = 0;
    if (src.mem) memcpy(&v, src.mem + src.offset + cell * (uint64_t)w, (size_t)w);
    else if (pread(fd, &v, (size_t)w, (off_t)(src.offset + cell * (uint64_t)w)) != (ssize_t)w) throw std::runtime_error("cannot read " + src.file);
    return v;
}

// Contiguous ranges of WHOLE strings balanced by symbol count (the reference's mt split, parsing_strategies.h:208-214,
// byte-balanced): boundary r is the end of the first string that ends at or after cell r*n/G. Fewer ranges than asked
// come back when the collection has fewer strings than ranks. -> cell offsets [b0=0, b1, ..., n]
inline std::vector<uint64_t> shard_bounds(const TextSource& src, int sym_bytes, int n_ranks) {
    const uint64_t w = (uint64_t)sym_bytes, n = src.bytes / w;
    int fd = -1;
    if (!src.mem) {
        fd = open(src.file.c_str(), O_RDONLY);
        if (fd < 0) throw std::runtime_error("cannot open " + src.file);
    }
    std::vector<uint64_t> b{0};
    try {
        const uint64_t sep = read_cell(src, fd, n - 1, sym_bytes);
        std::vector<unsigned char> win((size_t)(1u << 20) * w);
        for (int r = 1; r < n_ranks; r++) {
            uint64_t pos = std::max<uint64_t>((uint64_t)r * n / (uint64_t)n_ranks, b.back());
            uint64_t end = n;  // one past the separator that closes the string holding cell `pos`
            while (pos < n) {
                const uint64_t cnt = std::min<uint64_t>((uint64_t)1 << 20, n - pos);
                const unsigned char* p;
                if (src.mem) p = src.mem + src.offset + pos * w;
                else {
                    uint64_t got = 0;
                    while (got < cnt * w) {
                        const ssize_t rr = pread(fd, win.data() + got, cnt * w - got, (off_t)(src.offset + pos * w + got));
                        if (rr <= 0) throw std::runtime_error("cannot read " + src.file);
                        got += (uint64_t)rr;
                    }
                    p = win.data();
                }
                uint64_t k = 0;
                for (; k < cnt; k++) {
                    uint64_t v = 0;
                    memcpy(&v, p + k * w, (size_t)w);
                    if (v == sep) break;
                }
                if (k < cnt) { end = pos + k + 1; break; }
                pos += cnt;
            }
            if (end >= n) break;  // no further string boundary: the remaining ranks would be empty
            if (end > b.back()) b.push_back(end);
        }
    } catch (...) {
        if (fd >= 0) close(fd);
        throw;
    }
    if (fd >= 0) close(fd);
    b.push_back(n);
    return b;
}

// (stdio, not iostream: the library is also loaded into processes that carry another libstdc++, e.g. Python with torch)
inline void print_stats(const grlgpu_stats_t& s) {
    printf("Stats: \n");
    printf("  Smallest symbol               : %llu\n", (unsigned long long)s.min_sym);
    printf("  Greatest symbol               : %llu\n", (unsigned long long)s.max_sym);
    printf("  Number of symbols in the file : %llu\n", (unsigned long long)s.n_syms);
    printf("  Number of strings             : %llu\n", (unsigned long long)s.n_strings);
    printf("Parsing the text:    \n");
    fflush(stdout);
}
inline void print_round(const grlgpu_round_t& r) {
    printf("  Parsing round %llu\n", (unsigned long long)r.round);
    printf("    Stats:\n");
    printf("      Parsing phrases:                  %llu\n", (unsigned long long)r.n_phrases);
    printf("      Number of symbols in the phrases: %llu\n", (unsigned long long)r.dict_syms);
    printf("      Number of unsolved BWT blocks:    %llu\n", (unsigned long long)r.tot_phrases);
    printf("      Parse size:                       %llu\n", (unsigned long long)r.parse_len);
    printf("      Device time (ms):                 %g (text %g, dictionary %g, rewrite %g)\n", r.device_ms, r.text_pass_ms, r.dict_ms, r.rewrite_ms);
    fflush(stdout);
}

// storage of one level on the host, shared by the ranks of a multi-GPU run (each fills its own part)
struct LevelSink {
    bool wide = false, narrow_len = false;
    Level32 l32;
    Level l64;
    void prepare(const grlgpu_round_t& r, bool wide_) {
        wide = wide_;
        narrow_len = !wide && (r.n_in + r.parse_len < (1ull << 32));  // the run lengths of a level sum to at most n_in + parse_len
        if (!wide) {
            l32.alphabet = r.alphabet; l32.tot_phrases = r.tot_phrases;
            l32.rule_l.resize(r.tot_phrases); l32.rule_r.resize(r.tot_phrases); l32.has_hocc.resize(r.tot_phrases);
            l32.pre_sym.resize(r.n_pre_runs);
            if (narrow_len) l32.pre_len32.resize(r.n_pre_runs); else l32.pre_len.resize(r.n_pre_runs);
        } else {
            l64.alphabet = r.alphabet; l64.tot_phrases = r.tot_phrases;
            l64.rule_l.resize(r.tot_phrases); l64.rule_r.resize(r.tot_phrases); l64.has_hocc.resize(r.tot_phrases);
            l64.pre_sym.resize(r.n_pre_runs); l64.pre_len.resize(r.n_pre_runs);
        }
    }
};

// parks the context's current level (or level slice) and queues its copies into `sink` at the given element offsets.
// 32-bit device symbols into a 64-bit sink (a wide level followed by a narrower one) go through a widening copy.
inline void queue_level(const CtxHandle& ctx, FetchPool& pool, LevelSink& sink, uint64_t rank_off, uint64_t pre_off, std::vector<std::unique_ptr<RawBuf<uint32_t>>>& tmp32,
                        std::vector<std::function<void()>>& after) {
    grlgpu_level_ptrs_t lp;
    ctx.check("grlgpu_level_park", grlgpu_level_park(ctx.p, sink.narrow_len ? 4 : 8, &lp));
    if (!sink.wide) {
        if (lp.sym_bytes != 4) throw std::runtime_error("a 64-bit level reached the 32-bit sink");
        pool.enqueue(lp.device, sink.l32.rule_l.data() + rank_off, lp.rule_l, lp.tot * 4);
        pool.enqueue(lp.device, sink.l32.rule_r.data() + rank_off, lp.rule_r, lp.tot * 4);
        pool.enqueue(lp.device, sink.l32.has_hocc.data() + rank_off, lp.has_hocc, lp.tot);
        pool.enqueue(lp.device, sink.l32.pre_sym.data() + pre_off, lp.pre_sym, lp.n_pre * 4);
        if (sink.narrow_len) pool.enqueue(lp.device, sink.l32.pre_len32.data() + pre_off, lp.pre_len, lp.n_pre * 4);
        else pool.enqueue(lp.device, sink.l32.pre_len.data() + pre_off, lp.pre_len, lp.n_pre * 8);
        return;
    }
    pool.enqueue(lp.device, sink.l64.has_hocc.data() + rank_off, lp.has_hocc, lp.tot);
    pool.enqueue(lp.device, sink.l64.pre_len.data() + pre_off, lp.pre_len, lp.n_pre * 8);
    if (lp.sym_bytes == 8) {
        pool.enqueue(lp.device, sink.l64.rule_l.data() + rank_off, lp.rule_l, lp.tot * 8);
        pool.enqueue(lp.device, sink.l64.rule_r.data() + rank_off, lp.rule_r, lp.tot * 8);
        pool.enqueue(lp.device, sink.l64.pre_sym.data() + pre_off, lp.pre_sym, lp.n_pre * 8);
        return;
    }
    struct W { const void* src; uint64_t n; uint64_t* dst; };
    for (const W& wv : {W{lp.rule_l, lp.tot, sink.l64.rule_l.data() + rank_off}, W{lp.rule_r, lp.tot, sink.l64.rule_r.data() + rank_off},
                        W{lp.pre_sym, lp.n_pre, sink.l64.pre_sym.data() + pre_off}}) {
        tmp32.emplace_back(new RawBuf<uint32_t>(wv.n));
        uint32_t* t = tmp32.back()->data();
        pool.enqueue(lp.device, t, wv.src, wv.n * 4);
        uint64_t* dst = wv.dst;
        const uint64_t n = wv.n;
        after.push_back([t, dst, n] { for (uint64_t i = 0; i < n; i++) dst[i] = t[i]; });
    }
}

// first wide level: what was collected in 32-bit levels moves to 64-bit symbols
inline void widen_levels(ParseResult& res) {
    for (const Level32& s : res.levels32) {
        Level L;
        L.alphabet = s.alphabet; L.tot_phrases = s.tot_phrases;
        L.has_hocc.assign(s.has_hocc.begin(), s.has_hocc.end());
        if (!s.pre_len32.empty()) L.pre_len.assign(s.pre_len32.begin(), s.pre_len32.end());
        else L.pre_len.assign(s.pre_len.begin(), s.pre_len.end());
        L.rule_l.assign(s.rule_l.begin(), s.rule_l.end());
        L.rule_r.assign(s.rule_r.begin(), s.rule_r.end());
        L.pre_sym.assign(s.pre_sym.begin(), s.pre_sym.end());
        res.levels.push_back(std::move(L));
    }
    res.levels32.clear();
    res.wide = true;
}

// the collected levels in round order into res.levels32, or into res.levels from the first wide level on (every level then
// moves to 64-bit symbols)
inline void collect_levels(std::vector<std::unique_ptr<LevelSink>>& sinks, ParseResult& res) {
    res.wide = false;
    for (auto& s : sinks) {
        if (!s->wide) res.levels32.push_back(std::move(s->l32));
        else {
            if (!res.wide) widen_levels(res);
            res.levels.push_back(std::move(s->l64));
        }
    }
}

// every level kept on the device, copied to the host (the device induction is not going to consume them); drops them there
inline std::vector<Level32> fetch_kept_levels(const CtxHandle& ctx) {
    std::vector<Level32> out;
    for (int lv = 0; lv < grlgpu_kept_levels(ctx.p); lv++) {
        Level32 L;
        uint64_t A = 0, tot = 0, n_pre = 0;
        ctx.check("grlgpu_fetch_kept_level", grlgpu_fetch_kept_level(ctx.p, lv, &A, &tot, &n_pre, nullptr, nullptr, nullptr, nullptr, nullptr));
        L.alphabet = A; L.tot_phrases = tot;
        L.rule_l.resize(tot); L.rule_r.resize(tot); L.has_hocc.resize(tot); L.pre_sym.resize(n_pre); L.pre_len.resize(n_pre);
        ctx.check("grlgpu_fetch_kept_level", grlgpu_fetch_kept_level(ctx.p, lv, nullptr, nullptr, nullptr, L.rule_l.data(), L.rule_r.data(), L.has_hocc.data(), L.pre_sym.data(),
                                                                    (uint64_t*)L.pre_len.data()));
        out.push_back(std::move(L));
    }
    grlgpu_drop_kept(ctx.p);
    return out;
}

// n cells of `width` bytes each -> 64-bit values
inline void decode_cells(const unsigned char* raw, uint64_t n, uint32_t width, uint64_t* dst) {
    for (uint64_t i = 0; i < n; i++) {
        uint64_t v = 0;
        memcpy(&v, raw + i * width, width);
        dst[i] = v;
    }
}

// the sizes of a round's digest (the checksums are added by the caller)
inline RoundDigest digest_of(const grlgpu_round_t& r) {
    RoundDigest dg;
    dg.tot = r.tot_phrases; dg.n_pre = r.n_pre_runs; dg.parse_len = r.parse_len; dg.n_phrases = r.n_phrases; dg.dict_syms = r.dict_syms;
    return dg;
}

// header widths of the level-0 BWT (exact_ind_phase.cpp:274-276 with the level-0 dictionary: alphabet = max_sym+1+3,
// prev_alphabet = 0, max_sym_freq from collection_stats; SURVEY.md App. C)
inline void header_widths(const grlgpu_stats_t& stats, uint64_t& sb, uint64_t& fb) {
    sb = int_ceil((uint64_t)sym_width(stats.max_sym + 1 + 3), 8);
    fb = int_ceil((uint64_t)sym_width(stats.max_sym_freq), 8);
}

// the levels kept on the device -> level-0 BWT in res.bwt_dev; false (with the kept levels fetched into res.levels32) when the
// device cannot do it (size limits, memory): the caller then induces on the host
inline bool induce_on_device(const CtxHandle& ctx, ParseResult& res, const void* final_parse, uint64_t n_strings, int cell_bytes, bool verbose,
                             const OutputBuffers* ob = nullptr) {
    const auto t0 = std::chrono::steady_clock::now();
    uint64_t n_runs = 0;
    const int rc = grlgpu_induce(ctx.p, final_parse, n_strings, cell_bytes, res.stats.n_syms, &n_runs);
    if (rc == GRLGPU_OK) {
        const double compute_ms = ms_since(t0);
        res.bwt_dev.n = n_runs;
        res.dev_ind_compute_ms = compute_ms;
        if (ob && ob->packed) {  // .rl_bwt records packed on the device, straight into the caller's (pinned) buffer
            uint64_t sb = 0, fb = 0, nb = 0;
            header_widths(res.stats, sb, fb);
            const int st = grlgpu_fetch_bwt_packed(ctx.p, (int)sb, (int)fb, ob->packed, ob->packed_cap, &nb);
            if (st == GRLGPU_ERR_ARG && nb > ob->packed_cap) throw GpuError(GRLGPU_ERR_LIMIT, "the output buffer is too small: the .rl_bwt image has " + std::to_string(nb) + " bytes");
            ctx.check("grlgpu_fetch_bwt_packed", st);
            res.packed_bytes = nb;
            res.bwt_in_caller_buffers = true;
        } else if (ob && ob->sym && ob->len && ob->cap >= n_runs) {  // straight into the caller's (pinned) buffers
            ctx.check("grlgpu_fetch_bwt", grlgpu_fetch_bwt(ctx.p, ob->sym, ob->len));
            res.bwt_in_caller_buffers = true;
        } else {   // fresh pageable arrays: several copy threads, each staging (and first-touching) its own pieces
            res.bwt_dev.sym.alloc(n_runs);
            res.bwt_dev.len32.alloc(n_runs);
            const uint32_t *ds = nullptr, *dl = nullptr;
            uint64_t nr = 0;
            ctx.check("grlgpu_bwt_ptrs", grlgpu_bwt_ptrs(ctx.p, &ds, &dl, &nr));
            const int device = grlgpu_device_of(ctx.p);
            FetchPool pool(8);
            pool.enqueue(device, res.bwt_dev.sym.data(), ds, nr * 4);
            pool.enqueue(device, res.bwt_dev.len32.data(), dl, nr * 4);
            pool.wait_all();
        }
        grlgpu_drop_kept(ctx.p);
        res.induced_on_device = true;
        res.dev_ind_ms = ms_since(t0);
        if (verbose) { printf("  induction on the device: %.1f ms, %llu runs copied back in %.1f ms\n", compute_ms, (unsigned long long)n_runs, res.dev_ind_ms - compute_ms); fflush(stdout); }
        return true;
    }
    if (rc != GRLGPU_ERR_LIMIT && rc != GRLGPU_ERR_NOMEM) ctx.check("grlgpu_induce", rc);
    if (verbose) { printf("  (the device cannot hold the induction of this collection: %s; inducing on the host)\n", grlgpu_last_error(ctx.p)); fflush(stdout); }
    const int n_kept = grlgpu_kept_levels(ctx.p);  // the levels the failed attempt had not consumed yet are still there: all of them, it fails before consuming
    if (n_kept != (int)res.rounds.size()) throw GpuError(rc, std::string("grlgpu_induce: ") + grlgpu_strerror(rc) + " (" + grlgpu_last_error(ctx.p) + ")");
    res.levels32 = fetch_kept_levels(ctx);
    return false;
}

// ---------------------------------------------------------------- one GPU
inline ParseResult gpu_par_phase(const TextSource& src, int sym_bytes, int device, bool verbose, bool dev_induction = false, const OutputBuffers* ob = nullptr,
                                 size_t fetch_threads = 4) {
    ParseResult res;
    res.comm_kind = "single GPU";
    CtxHandle ctx(device, 0);
    res.h2d_ms = load_text(ctx, src, sym_bytes);
    auto t0 = std::chrono::steady_clock::now();
    ctx.check("grlgpu_stats", grlgpu_stats(ctx.p, &res.stats));
    if (verbose) print_stats(res.stats);
    FetchPool pool(fetch_threads);
    std::vector<std::unique_ptr<LevelSink>> sinks;
    std::vector<std::unique_ptr<RawBuf<uint32_t>>> tmp32;
    std::vector<std::function<void()>> after;
    for (;;) {
        grlgpu_round_t r;
        ctx.check("grlgpu_round", grlgpu_round(ctx.p, &r));
        RoundDigest dg = digest_of(r);
        ctx.check("grlgpu_level_checksum", grlgpu_level_checksum(ctx.p, dg.cs));
        res.digests.push_back(dg);
        if (dev_induction && r.sym_bytes == 4) {
            ctx.check("grlgpu_keep_level", grlgpu_keep_level(ctx.p));  // stays on the device for grlgpu_induce
        } else {
            if (dev_induction) {  // a wide level: the whole induction goes to the host; move what was kept so far
                dev_induction = false;
                for (Level32& L : fetch_kept_levels(ctx)) {
                    sinks.emplace_back(new LevelSink());
                    sinks.back()->l32 = std::move(L);
                }
            }
            // the copies of the previous level ran while this round computed; release its device arrays, then hand this level over
            pool.wait_all();
            ctx.check("grlgpu_fetch_wait", grlgpu_fetch_wait(ctx.p));
            const bool wide = res.wide || r.sym_bytes == 8;
            sinks.emplace_back(new LevelSink());
            sinks.back()->prepare(r, wide);
            res.wide = wide;
            queue_level(ctx, pool, *sinks.back(), 0, 0, tmp32, after);
        }
        if (verbose) print_round(r);
        res.rounds.push_back(r);
        if (r.done) {
            if (dev_induction) {
                res.par_ms = ms_since(t0);
                if (induce_on_device(ctx, res, nullptr, r.parse_len, (int)r.cell_bytes_out, verbose, ob)) return res;
            }
            std::vector<unsigned char> raw(r.parse_len * (uint64_t)r.cell_bytes_out);
            ctx.check("grlgpu_fetch_parse", grlgpu_fetch_parse(ctx.p, raw.data()));
            res.final_parse.resize(r.parse_len);
            decode_cells(raw.data(), r.parse_len, r.cell_bytes_out, res.final_parse.data());
            break;
        }
    }
    if (!res.levels32.empty()) {  // the device induction gave up at the end: its levels were fetched into levels32 already
        res.par_ms = ms_since(t0);
        return res;
    }
    pool.wait_all();
    ctx.check("grlgpu_fetch_wait", grlgpu_fetch_wait(ctx.p));
    for (auto& f : after) f();
    collect_levels(sinks, res);
    res.par_ms = ms_since(t0);
    return res;
}

// ---------------------------------------------------------------- several GPUs: one host thread per rank
struct HostBarrier {
    std::mutex m;
    std::condition_variable cv;
    int n, arrived = 0;
    uint64_t gen = 0;
    bool failed = false;
    explicit HostBarrier(int n_) : n(n_) {}
    void wait() {
        std::unique_lock<std::mutex> lk(m);
        if (failed) throw std::runtime_error("another rank failed");
        const uint64_t g = gen;
        if (++arrived == n) { arrived = 0; gen++; cv.notify_all(); }
        else cv.wait(lk, [&] { return gen != g || failed; });
        if (failed) throw std::runtime_error("another rank failed");
    }
    void abort() {
        std::lock_guard<std::mutex> lk(m);
        failed = true;
        cv.notify_all();
    }
};

enum CommKind { COMM_AUTO = 0, COMM_LOCAL = 1, COMM_NCCL = 2 };

// devices: one entry per rank (a device may repeat: several ranks then share it, and the exchange is the in-process one)
inline ParseResult gpu_par_phase_mg(const TextSource& src, int sym_bytes, const std::vector<int>& devices, int comm_kind, bool verbose, bool dev_induction = false,
                                    const OutputBuffers* ob = nullptr, size_t fetch_threads = 2) {
    const std::vector<uint64_t> bounds = shard_bounds(src, sym_bytes, (int)devices.size());
    const int G = (int)bounds.size() - 1;
    if (G <= 1) return gpu_par_phase(src, sym_bytes, devices.at(0), verbose, dev_induction, ob);
    bool distinct = true;
    for (int a = 0; a < G; a++)
        for (int b = a + 1; b < G; b++) distinct = distinct && devices[(size_t)a] != devices[(size_t)b];
    if (const char* e = getenv("GRLBWT_COMM")) comm_kind = !strcmp(e, "nccl") ? COMM_NCCL : !strcmp(e, "local") ? COMM_LOCAL : comm_kind;
    // auto: in-process ranks whose GPUs can address each other exchange by peer copies (copy engines at NVLink rate, no communicator
    // to set up: NCCL's costs ~1 s per process); NCCL when asked for, or when some pair of GPUs has no peer access
    bool all_peers = true;
    for (int a = 0; a < G; a++)
        for (int b = a + 1; b < G; b++) all_peers = all_peers && grlgpu_can_peer(devices[(size_t)a], devices[(size_t)b]) != 0;
    unsigned char nccl_id[128];
    bool use_nccl = comm_kind == COMM_NCCL || (comm_kind == COMM_AUTO && distinct && !all_peers);
    if (use_nccl && grlgpu_nccl_unique_id(nccl_id) != GRLGPU_OK) {
        if (comm_kind == COMM_NCCL) throw GpuError(GRLGPU_ERR_CUDA, "NCCL was requested but is not available");
        use_nccl = false;
    }
    if (use_nccl && !distinct) throw GpuError(GRLGPU_ERR_ARG, "NCCL needs one distinct GPU per rank");
    grlgpu_local_group* group = nullptr;
    if (!use_nccl && grlgpu_local_group_create(&group, G) != GRLGPU_OK) throw GpuError(GRLGPU_ERR_ARG, "cannot create the rank group");

    ParseResult res;
    res.n_ranks = G;
    HostBarrier bar(G);
    std::vector<std::string> errors((size_t)G);
    std::vector<int> err_status((size_t)G, 0);
    std::vector<std::unique_ptr<LevelSink>> sinks;
    std::vector<uint64_t> str_off((size_t)G + 1, 0);   // strings before each rank (filled after the stats)
    std::vector<std::array<uint64_t, 4>> cs_part((size_t)G);
    std::vector<uint64_t> xbytes((size_t)G, 0), local_strings((size_t)G, 0);
    std::vector<double> h2d((size_t)G, 0);
    const uint64_t w = (uint64_t)sym_bytes;
    const auto t_start = std::chrono::steady_clock::now();
    // device induction: rank 0's context adopts every level (the ranks copy their slices into it over NVLink / on the device)
    bool dev_ind = dev_induction;
    grlgpu_level_ptrs_t adopt{};
    double par_done_ms = 0;

    auto rank_main = [&](int me) {
        grlgpu_comm* comm = nullptr;
        try {
            CtxHandle ctx(devices[(size_t)me], 0);
            ctx.check("grlgpu_set_peers", grlgpu_set_peers(ctx.p, devices.data(), G));
            const auto t_c = std::chrono::steady_clock::now();
            int rc = use_nccl ? grlgpu_comm_create_nccl(&comm, nccl_id, me, G, devices[(size_t)me]) : grlgpu_comm_create_local(&comm, group, me, devices[(size_t)me]);
            if (rc != GRLGPU_OK) throw GpuError(rc, std::string("creating the exchange layer: ") + grlgpu_strerror(rc));
            if (verbose && me == 0) { printf("  exchange layer ready in %.1f ms\n", ms_since(t_c)); fflush(stdout); }
            TextSource shard = src;
            shard.offset = src.offset + bounds[(size_t)me] * w;
            shard.bytes = (bounds[(size_t)me + 1] - bounds[(size_t)me]) * w;
            h2d[(size_t)me] = load_text(ctx, shard, sym_bytes);
            grlgpu_stats_t gs;
            ctx.check("grlgpu_mg_stats", grlgpu_mg_stats(ctx.p, comm, &gs));
            {
                grlgpu_stats_t ls;
                ctx.check("grlgpu_stats", grlgpu_stats(ctx.p, &ls));
                local_strings[(size_t)me] = ls.n_strings;
            }
            if (me == 0) {
                res.stats = gs;
                if (verbose) print_stats(gs);
                char kind[128];
                grlgpu_comm_info(comm, nullptr, nullptr, nullptr, kind, sizeof(kind));
                res.comm_kind = kind;
            }
            bar.wait();
            if (me == 0) {
                for (int p = 0; p < G; p++) str_off[(size_t)p + 1] = str_off[(size_t)p] + local_strings[(size_t)p];
                res.final_parse.resize(gs.n_strings);
            }
            FetchPool pool(fetch_threads);
            std::vector<std::unique_ptr<RawBuf<uint32_t>>> tmp32;
            std::vector<std::function<void()>> after;
            for (;;) {
                grlgpu_round_t r;
                ctx.check("grlgpu_mg_round", grlgpu_mg_round(ctx.p, comm, &r));
                grlgpu_slice_t sl;
                ctx.check("grlgpu_mg_slice_info", grlgpu_mg_slice_info(ctx.p, &sl));
                ctx.check("grlgpu_mg_slice_checksum", grlgpu_mg_slice_checksum(ctx.p, cs_part[(size_t)me].data()));
                xbytes[(size_t)me] += sl.exchange_bytes;
                pool.wait_all();  // the previous level's copies ran during this round
                ctx.check("grlgpu_fetch_wait", grlgpu_fetch_wait(ctx.p));
                bar.wait();
                if (me == 0) {    // the level's host arrays, sized from the global counts every rank was told
                    RoundDigest dg = digest_of(r);
                    for (int p = 0; p < G; p++)
                        for (int k = 0; k < 4; k++) dg.cs[k] += cs_part[(size_t)p][(size_t)k];
                    res.digests.push_back(dg);
                    res.wide = res.wide || r.sym_bytes == 8;
                    sinks.emplace_back(new LevelSink());
                    sinks.back()->prepare(r, res.wide);
                    if (verbose) { print_round(r); printf("      Wall clock since start (ms):       %.1f\n", ms_since(t_start)); fflush(stdout); }
                    res.rounds.push_back(r);
                }
                if (dev_ind && me == 0) {
                    if (r.sym_bytes == 4) ctx.check("grlgpu_level_adopt", grlgpu_level_adopt(ctx.p, r.alphabet, r.tot_phrases, r.n_pre_runs, &adopt));
                    else {  // a wide level: the induction goes to the host; what rank 0 adopted so far moves into host levels
                        dev_ind = false;
                        std::unique_ptr<LevelSink> cur = std::move(sinks.back());
                        sinks.pop_back();
                        for (Level32& L : fetch_kept_levels(ctx)) {
                            sinks.emplace_back(new LevelSink());
                            sinks.back()->l32 = std::move(L);
                        }
                        sinks.push_back(std::move(cur));
                    }
                }
                bar.wait();
                if (dev_ind) {
                    grlgpu_level_ptrs_t lp;
                    ctx.check("grlgpu_level_park", grlgpu_level_park(ctx.p, 8, &lp));
                    struct C { char* dst; const void* src; uint64_t bytes; };
                    int rc = GRLGPU_OK;
                    for (const C& c : {C{(char*)adopt.rule_l + sl.rank_base * 4, lp.rule_l, lp.tot * 4}, C{(char*)adopt.rule_r + sl.rank_base * 4, lp.rule_r, lp.tot * 4},
                                       C{(char*)adopt.has_hocc + sl.rank_base, lp.has_hocc, lp.tot}, C{(char*)adopt.pre_sym + sl.pre_first * 4, lp.pre_sym, lp.n_pre * 4},
                                       C{(char*)adopt.pre_len + sl.pre_first * 8, lp.pre_len, lp.n_pre * 8}})
                        if (rc == GRLGPU_OK) rc = grlgpu_copy_dev(adopt.device, c.dst, lp.device, c.src, c.bytes);
                    if (rc != GRLGPU_OK) throw GpuError(rc, "copying a level slice to rank 0's device failed");
                    ctx.check("grlgpu_fetch_wait", grlgpu_fetch_wait(ctx.p));
                    bar.wait();  // the adopted level is complete before rank 0 adopts the next one
                } else
                    queue_level(ctx, pool, *sinks.back(), sl.rank_base, sl.pre_first, tmp32, after);
                if (r.done) {
                    std::vector<unsigned char> raw(sl.parse_len_local * (uint64_t)r.cell_bytes_out + 8);
                    ctx.check("grlgpu_fetch_parse", grlgpu_fetch_parse(ctx.p, raw.data()));
                    if (sl.parse_len_local != local_strings[(size_t)me]) throw std::runtime_error("the final parse of a rank is not one cell per string");
                    decode_cells(raw.data(), sl.parse_len_local, r.cell_bytes_out, res.final_parse.data() + str_off[(size_t)me]);
                    break;
                }
            }
            pool.wait_all();
            ctx.check("grlgpu_fetch_wait", grlgpu_fetch_wait(ctx.p));
            for (auto& f : after) f();
            bar.wait();
            grlgpu_comm_destroy(comm);
            comm = nullptr;
            if (me == 0) par_done_ms = ms_since(t_start);
            if (dev_ind && me == 0) {  // every level sits in this context, the final parse of all ranks in res.final_parse (string order)
                if (induce_on_device(ctx, res, res.final_parse.data(), res.final_parse.size(), 8, verbose, ob)) sinks.clear();
            }
        } catch (const GpuError& e) {
            errors[(size_t)me] = e.what();
            err_status[(size_t)me] = e.status;
            bar.abort();
            if (group) grlgpu_local_group_abort(group);
            if (comm) grlgpu_comm_destroy(comm);
        } catch (const std::exception& e) {
            errors[(size_t)me] = e.what();
            err_status[(size_t)me] = -100;
            bar.abort();
            if (group) grlgpu_local_group_abort(group);
            if (comm) grlgpu_comm_destroy(comm);
        }
    };
    std::vector<std::thread> th;
    for (int r = 0; r < G; r++) th.emplace_back(rank_main, r);
    for (auto& t : th) t.join();
    if (group) grlgpu_local_group_destroy(group);
    // the first real failure (not the "another rank failed" echoes it caused)
    int first_bad = -1;
    for (int r = 0; r < G; r++)
        if (err_status[(size_t)r] && (first_bad < 0 || (errors[(size_t)first_bad].find("another rank failed") != std::string::npos &&
                                                         errors[(size_t)r].find("another rank failed") == std::string::npos)))
            first_bad = r;
    if (first_bad >= 0) throw GpuError(err_status[(size_t)first_bad], "rank " + std::to_string(first_bad) + ": " + errors[(size_t)first_bad]);
    if (!res.induced_on_device && res.levels32.empty()) collect_levels(sinks, res);
    for (int r = 0; r < G; r++) { res.exchange_bytes += xbytes[(size_t)r]; res.h2d_ms = std::max(res.h2d_ms, h2d[(size_t)r]); }
    res.par_ms = par_done_ms - res.h2d_ms;
    return res;
}

}  // namespace grlbwt
