"""Reference answers for the search with mismatches (fm_query -k, fm_query_gpu -k, GrlGpu.fm_approx_*).

An occurrence of P with d mismatches is (k, p, d): the window S_k[p .. p + m) lies inside string k and differs from P in exactly
d <= max_mismatches positions. A pattern cell that is the separator or a symbol absent from the collection never matches.
Two oracles: every in-string window of a small collection (naive), and the pigeonhole filter at scale: a window with at most k
mismatches holds one of k + 1 pieces of P exactly, so the candidates are the exact occurrences of the pieces (fm_oracle.Text)."""
import numpy as np

from fm_oracle import Text


def naive(t: Text, pat, kmax):
    """sorted list of (k, p, d) over every window of the collection, vectorised over the windows"""
    return _as_triples(t, *_windows_within(t, pat, kmax))


def naive_counts(t: Text, pat, kmax):
    """the number of occurrences with d = 0 .. kmax mismatches, from every window"""
    return np.bincount(_windows_within(t, pat, kmax)[1], minlength=kmax + 1)


def _windows_within(t, pat, kmax):
    pat = np.asarray(pat, np.uint64)
    if not hasattr(t, "_windows"):   # per collection: its cells as uint64, separator counts, in-string windows per length
        t._a64, t._is_sep, t._windows = t.arr.astype(np.uint64), np.concatenate(([0], np.cumsum(t.arr == t.sep))), {}
    a, m = t._a64, pat.size
    if m == 0 or m > a.size:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    if m not in t._windows:
        x = np.arange(a.size - m + 1)
        t._windows[m] = x[t._is_sep[x + m] == t._is_sep[x]]   # no separator inside the window
    x = t._windows[m]
    dist = np.zeros(x.size, np.int64)
    for i in range(m):
        dist += a[x + i] != pat[i]
    keep = dist <= kmax
    return x[keep], dist[keep]


def pigeonhole(t: Text, pat, kmax):
    """the same list from the exact occurrences of k + 1 pieces of P, each candidate verified"""
    pat = np.asarray(pat, np.uint64)
    m = pat.size
    cuts = np.linspace(0, m, kmax + 2).astype(int)
    cand = set()
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        if hi > lo:
            for k, p in t.occurrences(pat[lo:hi]):
                if p >= lo:
                    cand.add(int(t.starts[k]) + p - lo)
    a, out_x, out_d = t.arr, [], []
    for x in sorted(cand):
        w = a[x:x + m]
        if w.size == m and not (w == t.sep).any():
            d = int((w.astype(np.uint64) != pat).sum())
            if d <= kmax:
                out_x.append(x)
                out_d.append(d)
    return _as_triples(t, np.asarray(out_x, np.int64), np.asarray(out_d, np.int64))


def _as_triples(t, x, d):
    k = np.searchsorted(t.ends, x)
    return sorted(zip(k.tolist(), (x - t.starts[k]).tolist(), d.tolist()))


def mutate(rng, windows, alpha, n_subs):
    """copies of the windows (2-d array) with n_subs[i] random positions of row i replaced by another symbol of alpha"""
    out = windows.copy()
    for i in range(out.shape[0]):
        for j in rng.choice(out.shape[1], int(n_subs[i]), replace=False):
            others = alpha[alpha != out[i, j]]
            if others.size:
                out[i, j] = rng.choice(others)
    return out


def patterns(t: Text, rng, n_win=30, n_rand=15, max_len=10):
    """windows of the strings with 0 to 2 substitutions, random patterns, and patterns with the separator or an absent symbol in
    them (lists of ints, each non-empty, of at most max_len cells)"""
    a, out = t.arr, []
    lens = t.ends - t.starts
    alpha = np.unique(a[a != t.sep]).astype(np.uint64)
    nonempty = np.flatnonzero(lens > 0)
    for _ in range(n_win if nonempty.size else 0):
        k = int(rng.choice(nonempty))
        m = int(rng.integers(1, min(max_len, lens[k]) + 1))
        p = int(rng.integers(0, lens[k] - m + 1))
        w = a[t.starts[k] + p: t.starts[k] + p + m].astype(np.uint64)[None, :]
        out.append(mutate(rng, w, alpha, [rng.integers(0, min(2, m) + 1)])[0].tolist())
    if alpha.size:
        for _ in range(n_rand):
            out.append(rng.choice(alpha, size=int(rng.integers(1, 7))).tolist())
        present = set(np.unique(a).tolist())
        absent = next(c for c in range(t.sep + 1, t.sep + 10**6) if c not in present)
        if absent <= np.iinfo(a.dtype).max:
            out += [[absent], [int(alpha[0]), absent], [absent, int(alpha[-1]), int(alpha[0])]]
        out += [[int(alpha[0]), t.sep, int(alpha[-1])], [t.sep]]   # only in the binding: the tools' files cannot hold the separator
    return out


def parse_output(out):
    """tool output with -k -> list of (count, [(k, p, d), ...] in the order printed)"""
    res = []
    for line in out.decode().splitlines():
        f = line.split()
        res.append((int(f[0]), [tuple(int(x) for x in e.split(":")) for e in f[1:]]))
    return res
