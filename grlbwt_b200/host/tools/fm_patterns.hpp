// Shared pieces of the search tools fm_query (host) and fm_query_gpu (device): the patterns file and the output lines; and the
// requests file of the extract tools fm_extract (host) and fm_extract_gpu (device).
#pragma once
#include <cstdint>
#include <cstdio>
#include <stdexcept>
#include <string>
#include <vector>

namespace grlbwt {

// patterns in grlBWT's input format: cells of w little-endian bytes, each pattern ended by the index's separator (a last pattern
// without one still counts). cells = the patterns' cells without separators, off = n_pat + 1 offsets into it. An empty pattern
// is an error.
inline void read_patterns(const std::string& path, int w, uint64_t sep, std::vector<uint64_t>& cells, std::vector<uint64_t>& off) {
    if (w != 1 && w != 2 && w != 4 && w != 8) throw std::runtime_error("the cell width must be 1, 2, 4 or 8");
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) throw std::runtime_error("cannot open " + path);
    std::vector<unsigned char> raw;
    unsigned char buf[1 << 16];
    for (size_t got; (got = fread(buf, 1, sizeof(buf), f)) > 0;) raw.insert(raw.end(), buf, buf + got);
    fclose(f);
    if (raw.size() % (size_t)w) throw std::runtime_error(path + " is not a whole number of " + std::to_string(w) + "-byte cells");
    cells.clear();
    off.assign(1, 0);
    for (size_t a = 0; a < raw.size(); a += (size_t)w) {
        uint64_t v = 0;
        for (int b = 0; b < w; b++) v |= (uint64_t)raw[a + (size_t)b] << (8 * b);
        if (v != sep) { cells.push_back(v); continue; }
        if (cells.size() == off.back()) throw std::runtime_error("pattern " + std::to_string(off.size() - 1) + " is empty");
        off.push_back(cells.size());
    }
    if (cells.size() != off.back()) off.push_back(cells.size());
}

// requests of the extract tools fm_extract (host) and fm_extract_gpu (device): a text file, one request per line, "k", "k from" or
// "k from len" in decimal, separated by spaces or tabs; a missing from is 0, a missing len means to the end of the string (len =
// UINT64_MAX). Any other line, a number beyond 64 bits or k >= n_strings is an error.
inline void read_requests(const std::string& path, uint64_t n_strings, std::vector<uint64_t>& k, std::vector<uint64_t>& from, std::vector<uint64_t>& len) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) throw std::runtime_error("cannot open " + path);
    std::string raw;
    char buf[1 << 16];
    for (size_t got; (got = fread(buf, 1, sizeof(buf), f)) > 0;) raw.append(buf, got);
    fclose(f);
    k.clear();
    from.clear();
    len.clear();
    size_t a = 0;
    for (uint64_t line = 1; a < raw.size(); line++) {
        size_t e = raw.find('\n', a);
        if (e == std::string::npos) e = raw.size();
        uint64_t v[3] = {0, 0, UINT64_MAX};
        int n_v = 0;
        for (size_t i = a; i < e;) {
            if (raw[i] == ' ' || raw[i] == '\t') { i++; continue; }
            bool ok = n_v < 3 && raw[i] >= '0' && raw[i] <= '9';
            uint64_t x = 0;
            for (; ok && i < e && raw[i] >= '0' && raw[i] <= '9'; i++) {
                const uint64_t d = (uint64_t)(raw[i] - '0');
                ok = x <= (UINT64_MAX - d) / 10;
                x = x * 10 + d;
            }
            if (!ok || (i < e && raw[i] != ' ' && raw[i] != '\t'))
                throw std::runtime_error(path + ", line " + std::to_string(line) + ": expected \"k\", \"k from\" or \"k from len\" in decimal");
            v[n_v++] = x;
        }
        if (n_v == 0) throw std::runtime_error(path + ", line " + std::to_string(line) + ": expected \"k\", \"k from\" or \"k from len\" in decimal");
        if (v[0] >= n_strings)
            throw std::runtime_error(path + ", line " + std::to_string(line) + ": string " + std::to_string(v[0]) + " does not exist (the BWT has " +
                                     std::to_string(n_strings) + " strings)");
        k.push_back(v[0]);
        from.push_back(v[1]);
        len.push_back(v[2]);
        a = e + 1;
    }
}

// one output line: the count, then " k:p" per occurrence in row order, or " k:p:d" with the mismatches d of each (search with -k)
template <class T>
inline void put_line(std::string& out, uint64_t count, const T* k, const T* p, const uint8_t* d = nullptr) {
    out += std::to_string(count);
    if (k)
        for (uint64_t o = 0; o < count; o++) {
            out += ' '; out += std::to_string(k[o]); out += ':'; out += std::to_string(p[o]);
            if (d) { out += ':'; out += std::to_string(d[o]); }
        }
    out += '\n';
}
// the -k argument of the search tools: 0 to 3 mismatches
inline uint32_t parse_mismatches(const char* s) {
    if (s[0] < '0' || s[0] > '3' || s[1]) throw std::runtime_error(std::string("-k takes 0, 1, 2 or 3 mismatches, not \"") + s + "\"");
    return (uint32_t)(s[0] - '0');
}
inline void flush_out(std::string& out, bool force) {
    if (!force && out.size() < (1u << 20)) return;
    fwrite(out.data(), 1, out.size(), stdout);
    out.clear();
}

}  // namespace grlbwt
