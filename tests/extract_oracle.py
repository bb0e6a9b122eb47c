"""Reference answers for extract (fm_extract, fm_extract_gpu, GrlGpu.fm_extract): numpy slices of the collection itself.

A request is (k, from, len) with from and len optional (None): S_k[from .. min(from + len, |S_k|)), the whole string without them."""
import numpy as np

U32_MAX = (1 << 32) - 1


def requests(t, rng, n_rand=40):
    """random requests over the strings of a fm_oracle.Text, and the edge cases: whole strings, from only, from at the string's end
    and beyond, len 0, the empty strings -> list of (k, from or None, len or None)"""
    lens = t.ends - t.starts
    N = lens.size
    out = []
    for _ in range(n_rand):
        k = int(rng.integers(0, N))
        out.append((k, int(rng.integers(0, lens[k] + 4)), int(rng.integers(0, lens[k] + 4))))
    for k in rng.choice(N, size=min(N, 20), replace=False).tolist():
        out += [(k, None, None), (k, int(rng.integers(0, lens[k] + 1)), None), (k, int(lens[k]), None), (k, int(lens[k]) + 5, 3),
                (k, 0, 0), (k, int(lens[k]) // 2, 0), (k, 0, U32_MAX)]
    out += [(int(k), None, None) for k in np.flatnonzero(lens == 0)[:20]]
    return out


def expected(t, reqs):
    """the substring of every request, as arrays of the collection's dtype"""
    res = []
    for k, f, m in reqs:
        a, b = int(t.starts[k]), int(t.ends[k])
        lo = a + (f or 0)
        hi = b if m is None else min(b, lo + m)
        res.append(t.arr[lo:hi] if lo < hi else t.arr[:0])
    return res


def requests_file(path, reqs):
    """the text form the tools read: "k", "k from" or "k from len" per line"""
    lines = []
    for k, f, m in reqs:
        lines.append(" ".join(str(x) for x in ([k] if f is None and m is None else [k, f or 0] if m is None else [k, f or 0, m])))
    with open(path, "w") as fh:
        fh.write("\n".join(lines) + "\n")


def as_arrays(reqs):
    """(str_id, start, length) arrays for GrlGpu.fm_extract: a missing len is UINT32_MAX, which also means to the end"""
    return (np.array([k for k, _, _ in reqs], np.uint64), np.array([f or 0 for _, f, _ in reqs], np.uint64),
            np.array([U32_MAX if m is None else m for _, _, m in reqs], np.uint64))


def low_bytes(arr, w):
    """the cells of width w that keep each symbol's low bytes (reverse_bwt's put_cell)"""
    mask = np.uint64((1 << (8 * w)) - 1)
    return (arr.astype(np.uint64) & mask).astype({1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}[w])


def tool_output(t, reqs, w):
    """what fm_extract writes: each substring followed by the separator, cells of width w"""
    sep = np.array([t.sep], t.arr.dtype)
    parts = []
    for x in expected(t, reqs):
        parts += [x, sep]
    return low_bytes(np.concatenate(parts) if parts else t.arr[:0], w).tobytes()
