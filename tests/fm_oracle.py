"""Reference answers for the FM-index searches (fm_query, fm_query_gpu, GrlGpu.fm_*): a naive find over the collection itself.

A collection is one array whose strings each end with the separator (its smallest symbol). An occurrence of P is (k, p) with
S_k[p .. p + len(P)) = P; a pattern containing the separator has none."""
import os
import subprocess

import numpy as np

from oracle import oracle as O


def image_of(arr):
    """the .rl_bwt image of a collection, built by the oracle (no device)"""
    o = O.Oracle(arr)
    o.par_phase()
    syms, lens, sb, fb = o.ind_phase()
    o.close()
    return O.rl_bwt_bytes(syms, lens, sb, fb), syms


class Text:
    def __init__(self, arr):
        self.arr = np.ascontiguousarray(arr)
        self.sep = int(arr[-1])
        self.ends = np.flatnonzero(self.arr == self.sep)
        self.starts = np.concatenate(([0], self.ends[:-1] + 1))

    def occurrences(self, pat):
        """sorted list of (k, p)"""
        pat = np.asarray(pat, dtype=np.uint64)
        m, a = pat.size, self.arr
        if m == 0 or (pat == self.sep).any() or m > a.size:
            return []
        cand = np.flatnonzero(a[: a.size - m + 1] == pat[0].astype(a.dtype) if pat[0] <= np.iinfo(a.dtype).max else np.zeros(0, np.int64))
        for i in range(1, m):
            if cand.size == 0:
                break
            if pat[i] > np.iinfo(a.dtype).max:
                return []
            cand = cand[a[cand + i] == pat[i]]
        k = np.searchsorted(self.ends, cand)   # the string holding position x: the first separator at or after it
        return sorted(zip(k.tolist(), (cand - self.starts[k]).tolist()))

    def patterns(self, rng, n_hits=40, n_rand=40, max_len=12):
        """sampled substrings, random patterns, single symbols, whole strings and an absent symbol (lists of ints, each non-empty)"""
        a, out = self.arr, []
        lens = self.ends - self.starts
        nonempty = np.flatnonzero(lens > 0)
        if nonempty.size:
            for _ in range(n_hits):
                k = int(rng.choice(nonempty))
                m = int(rng.integers(1, min(max_len, lens[k]) + 1))
                p = int(rng.integers(0, lens[k] - m + 1))
                out.append(a[self.starts[k] + p: self.starts[k] + p + m].astype(np.uint64).tolist())
            for k in rng.choice(nonempty, size=min(5, nonempty.size), replace=False):
                out.append(a[self.starts[k]: self.ends[k]].astype(np.uint64).tolist())
        alpha = np.unique(a[a != self.sep]).astype(np.uint64)
        if alpha.size:
            for _ in range(n_rand):
                out.append(rng.choice(alpha, size=int(rng.integers(1, 7))).tolist())
            out += [[int(c)] for c in alpha[:50]]
        present = set(np.unique(a).tolist())
        absent = next(c for c in range(self.sep + 1, self.sep + 10**6) if c not in present)
        if absent <= np.iinfo(a.dtype).max:
            out.append([absent])
            if alpha.size:
                out.append([int(alpha[0]), absent])
        return out


def patterns_file(path, pats, sep, w):
    """grlBWT's input format: each pattern followed by the separator"""
    cells = []
    for p in pats:
        cells += list(p) + [sep]
    np.asarray(cells, dtype=np.uint64).astype({1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}[w]).tofile(path)


def run_tool(tool, rl, pats_path, w, locate):
    cmd = [tool, str(rl), str(pats_path), "-a", str(w)] + (["-l"] if locate else [])
    r = subprocess.run(cmd, capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    return r.stdout


def parse_output(out):
    """tool output -> list of (count, [(k, p), ...] in the order printed)"""
    res = []
    for line in out.decode().splitlines():
        f = line.split()
        res.append((int(f[0]), [tuple(int(x) for x in t.split(":")) for t in f[1:]]))
    return res


def lib(name):
    import grlbwt_b200 as G
    return os.path.join(G.LIB_DIR, name)
