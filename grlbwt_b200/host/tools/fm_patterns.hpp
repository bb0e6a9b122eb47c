// Shared pieces of the search tools fm_query (host) and fm_query_gpu (device): the patterns file and the output lines.
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

// one output line: the count, then " k:p" per occurrence in row order
template <class T>
inline void put_line(std::string& out, uint64_t count, const T* k, const T* p) {
    out += std::to_string(count);
    if (k)
        for (uint64_t o = 0; o < count; o++) { out += ' '; out += std::to_string(k[o]); out += ':'; out += std::to_string(p[o]); }
    out += '\n';
}
inline void flush_out(std::string& out, bool force) {
    if (!force && out.size() < (1u << 20)) return;
    fwrite(out.data(), 1, out.size(), stdout);
    out.clear();
}

}  // namespace grlbwt
