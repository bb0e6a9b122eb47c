// Shared pieces of the .rl_bwt consumer tools (fresh equivalents of the reference's scripts/*.cpp, which need
// SDSL wavelet trees): a run-length BWT held as arrays, and LF-mapping over it with per-run rank prefixes and a
// binary search on run starts (O(log r) per step, any symbol width).
#pragma once
#include <algorithm>
#include <cstdint>
#include <exception>
#include <iostream>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

#include "../rl_bwt_io.hpp"

namespace grlbwt {

struct RlBwt {
    RunList runs;
    uint64_t sb = 0, fb = 0, n = 0;
    std::vector<uint64_t> start;      // start[i] = position of run i; start[r] = n
    std::vector<uint64_t> before;     // before[i] = occurrences of runs.sym[i] in runs 0..i-1
    std::map<uint64_t, uint64_t> C;   // C[c] = number of symbols smaller than c
    uint64_t sep = 0, n_strings = 0;

    explicit RlBwt(const std::string& path) {
        read_rl_bwt(path, runs, sb, fb);
        const size_t r = runs.size();
        start.resize(r + 1);
        before.resize(r);
        std::map<uint64_t, uint64_t> cnt;
        uint64_t max_sym = 0;
        for (size_t i = 0; i < r; i++) max_sym = std::max(max_sym, runs.sym[i]);
        if (max_sym < (1ull << 26)) {  // dense counters: one array access per run instead of a tree walk (billions of runs at full size)
            std::vector<uint64_t> dense(max_sym + 1, 0);
            for (size_t i = 0; i < r; i++) {
                start[i] = n;
                before[i] = dense[runs.sym[i]];
                dense[runs.sym[i]] += runs.len[i];
                n += runs.len[i];
            }
            for (uint64_t c = 0; c <= max_sym; c++)
                if (dense[c]) cnt[c] = dense[c];
        } else {
            for (size_t i = 0; i < r; i++) {
                start[i] = n;
                before[i] = cnt[runs.sym[i]];
                cnt[runs.sym[i]] += runs.len[i];
                n += runs.len[i];
            }
        }
        start[r] = n;
        uint64_t acc = 0;
        for (auto& kv : cnt) { C[kv.first] = acc; acc += kv.second; }
        if (!cnt.empty()) { sep = cnt.begin()->first; n_strings = cnt.begin()->second; }  // the separator is the smallest symbol
    }
    // symbol at position i and the row LF(i) = C[c] + rank_c(i)
    std::pair<uint64_t, uint64_t> lf(uint64_t i) const {
        const size_t k = (size_t)(std::upper_bound(start.begin(), start.end(), i) - start.begin()) - 1;
        const uint64_t c = runs.sym[k];
        return {c, C.at(c) + before[k] + (i - start[k])};
    }

    // ---- search (fm_query): per-symbol run lists, built by index_runs() ----
    std::vector<uint64_t> by_sym;                                  // run indices in (symbol, run index) order
    std::map<uint64_t, std::pair<uint64_t, uint64_t>> slice;       // symbol -> its range [lo, hi) of by_sym
    std::vector<uint64_t> c_val, c_sym;                            // C[c] and c, in symbol order
    void index_runs() {
        const size_t r = runs.size();
        by_sym.resize(r);
        uint64_t max_sym = 0;
        for (size_t i = 0; i < r; i++) max_sym = std::max(max_sym, runs.sym[i]);
        if (max_sym < (1ull << 26)) {  // counting sort by symbol
            std::vector<uint64_t> first(max_sym + 2, 0);
            for (size_t i = 0; i < r; i++) first[runs.sym[i] + 1]++;
            for (uint64_t c = 0; c <= max_sym; c++) first[c + 1] += first[c];
            std::vector<uint64_t> at(first.begin(), first.end() - 1);
            for (size_t i = 0; i < r; i++) by_sym[at[runs.sym[i]]++] = i;
        } else {
            for (size_t i = 0; i < r; i++) by_sym[i] = i;
            std::stable_sort(by_sym.begin(), by_sym.end(), [&](uint64_t a, uint64_t b) { return runs.sym[a] < runs.sym[b]; });
        }
        for (size_t q = 0; q < r;) {
            size_t e = q;
            while (e < r && runs.sym[by_sym[e]] == runs.sym[by_sym[q]]) e++;
            slice[runs.sym[by_sym[q]]] = {q, e};
            q = e;
        }
        for (auto& kv : C) { c_sym.push_back(kv.first); c_val.push_back(kv.second); }
    }
    // rank_c(BWT, i) for i in [0, n]: from the run holding i, or the last run of c before it
    uint64_t rank(uint64_t c, uint64_t i) const {
        const size_t k = (size_t)(std::upper_bound(start.begin(), start.end(), i) - start.begin()) - 1;  // i = n: k = r
        if (k < runs.size() && runs.sym[k] == c) return before[k] + (i - start[k]);
        const auto sl = slice.find(c);
        if (sl == slice.end()) return 0;
        const auto lo = by_sym.begin() + (long)sl->second.first;
        const size_t m = (size_t)(std::lower_bound(lo, by_sym.begin() + (long)sl->second.second, (uint64_t)k) - lo);
        if (m == 0) return 0;
        const uint64_t q = *(lo + (long)(m - 1));
        return before[q] + runs.len[q];
    }
    // rows [sp, ep) whose suffix starts with P; a pattern without occurrence (the separator or an absent symbol in it, or an empty
    // interval) gives sp = ep = 0, as the device search does
    std::pair<uint64_t, uint64_t> count(const uint64_t* P, size_t m) const {
        uint64_t sp = 0, ep = n;
        for (size_t a = m; a-- > 0;) {
            const auto it = C.find(P[a]);
            if (P[a] == sep || it == C.end()) return {0, 0};
            sp = it->second + rank(P[a], sp);
            ep = it->second + rank(P[a], ep);
            if (sp >= ep) return {0, 0};
        }
        return {sp, ep};
    }
    // search with at most k substitutions: every distinct string Q with Hamming(P, Q) <= k that occurs, as its rows [sp, ep) and
    // d = Hamming(P, Q), by ascending sp. A depth-first backward search over k + 1 frames, frame d the state after d substitutions
    // (cells 0 .. t - 1 still to match, the interval so far, the next symbol to substitute), as the device search does. A pattern
    // cell that is the separator or an absent symbol never matches; substitutions use every symbol but the separator.
    struct Hit { uint64_t sp, ep; uint32_t d; };
    std::vector<Hit> approx_count(const uint64_t* P, size_t m, uint32_t k) const {
        // the candidates of a frame: the symbols of the runs [sp, ep) spans when they are fewer than the alphabet (narrow intervals
        // of large alphabets), else every symbol
        struct Frame { size_t t; uint64_t sp, ep; size_t cur; std::vector<uint64_t> cand; };
        auto candidates = [&](uint64_t sp, uint64_t ep) {
            const size_t a = (size_t)(std::upper_bound(start.begin(), start.end(), sp) - start.begin()) - 1;
            const size_t b = (size_t)(std::lower_bound(start.begin(), start.end(), ep) - start.begin());
            if (b - a >= c_sym.size()) return c_sym;
            std::vector<uint64_t> c(runs.sym.begin() + (long)a, runs.sym.begin() + (long)b);
            std::sort(c.begin(), c.end());
            c.erase(std::unique(c.begin(), c.end()), c.end());
            return c;
        };
        std::vector<Hit> hits;
        if (m >= n) return hits;  // a window inside a string has fewer cells than the BWT has rows
        std::vector<Frame> f;
        f.push_back({m, 0, n, 0, k ? candidates(0, n) : std::vector<uint64_t>()});
        while (!f.empty()) {
            Frame& F = f.back();
            const uint32_t d = (uint32_t)(f.size() - 1);
            if (F.t == 0) {
                hits.push_back({F.sp, F.ep, d});
                f.pop_back();
                continue;
            }
            const uint64_t own = P[F.t - 1];
            if (d < k) {
                uint64_t sp = 0, ep = 0;
                while (F.cur < F.cand.size() && sp == ep) {
                    const uint64_t c = F.cand[F.cur++];
                    if (c == sep || c == own) continue;
                    sp = C.at(c) + rank(c, F.sp);
                    ep = C.at(c) + rank(c, F.ep);
                }
                if (sp < ep) {
                    const size_t t = F.t - 1;
                    f.push_back({t, sp, ep, 0, d + 1 < k && t ? candidates(sp, ep) : std::vector<uint64_t>()});
                    continue;
                }
            }
            const auto it = C.find(own);
            if (own == sep || it == C.end()) { f.pop_back(); continue; }
            const uint64_t sp = it->second + rank(own, F.sp), ep = it->second + rank(own, F.ep);
            if (sp >= ep) { f.pop_back(); continue; }
            F.t--;
            F.sp = sp;
            F.ep = ep;
            F.cur = 0;
            F.cand = d < k && F.t ? candidates(sp, ep) : std::vector<uint64_t>();
        }
        std::sort(hits.begin(), hits.end(), [](const Hit& a, const Hit& b) { return a.sp < b.sp; });
        return hits;
    }
    // psi(j) = LF^-1(j): the c of F row j, then the run of c that holds its (j - C[c])-th occurrence
    uint64_t psi(uint64_t j) const {
        const size_t d = (size_t)(std::upper_bound(c_val.begin(), c_val.end(), j) - c_val.begin()) - 1;
        const uint64_t x = j - c_val[d];
        const auto sl = slice.at(c_sym[d]);
        const auto lo = by_sym.begin() + (long)sl.first, hi = by_sym.begin() + (long)sl.second;
        const uint64_t q = *(std::upper_bound(lo, hi, x, [&](uint64_t v, uint64_t run) { return v < before[run]; }) - 1);
        return start[q] + (x - before[q]);
    }
    // occurrence at row j: string k (row k < n_strings is $_k, reached by psi) and offset p (LF steps to a separator)
    std::pair<uint64_t, uint64_t> locate(uint64_t j) const {
        uint64_t p = 0, r = j;
        for (auto e = lf(r); e.first != sep; e = lf(r = e.second))
            if (++p > n) throw std::runtime_error("the file is ill formed (an LF cycle without separator)");
        uint64_t k = j, f = 0;
        do {
            if (++f > n) throw std::runtime_error("the file is ill formed (an LF cycle without separator)");
            k = psi(k);
        } while (k >= n_strings);
        return {k, p};
    }

    // ---- extract (fm_extract) ----
    // S_k for k < n_strings: walked backwards by LF from row k, as reverse_bwt does. The walk ends within n steps for any run list:
    // the LF cycle of row k holds the separator row LF^-1(k).
    std::vector<uint64_t> string_of(uint64_t k) const {
        std::vector<uint64_t> s;
        for (auto e = lf(k); e.first != sep; e = lf(e.second)) s.push_back(e.first);
        std::reverse(s.begin(), s.end());
        return s;
    }
    // the cells [from, e) of S_k[from .. e) in a string of length L: e = min(from + len, L) without overflow, empty when from >= L
    static std::pair<uint64_t, uint64_t> clamp(uint64_t L, uint64_t from, uint64_t len) {
        if (from >= L) return {0, 0};
        return {from, len > L - from ? L : from + len};
    }
};

inline void put_cell(std::vector<unsigned char>& out, uint64_t v, int width) {
    for (int b = 0; b < width; b++) out.push_back((unsigned char)(v >> (8 * b)));
}

}  // namespace grlbwt

// a malformed input (bad header, truncated record) ends the tool with a message and status 1, not an abort
#define GRL_TOOL_MAIN(fn)                                             \
    int main(int argc, char** argv) {                                 \
        try { return fn(argc, argv); }                                \
        catch (const std::exception& e) { std::cerr << "Error: " << e.what() << std::endl; return 1; } \
    }
