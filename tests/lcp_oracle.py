"""Reference answers for the LCP array (fm_lcp, fm_lcp_gpu, GrlGpu.fm_lcp), independent of both tools.

The row order and the (k, p) of every row come from the .rl_bwt image alone: a stable argsort of the expanded BWT gives LF, and
walking LF from each row k < N ($_k, position L_k) down to the row whose symbol is the separator (position 0) names every row of
string k. Each LCP value is then found by comparing the two suffixes of the original collection directly, a separator never
matching (itself included). check_order ties that order to the text: for every j >= 1 the suffixes of rows j - 1 and j agree on
their first LCP[j] cells, and the next cell of row j - 1 is smaller than row j's unless one of the two is a separator."""
import numpy as np

from fm_oracle import Text
from grlbwt_b200.api import parse_rl_bwt


class Rows:
    """bwt (expanded), sep, N, and for every row its string k and offset p, from the image"""

    def __init__(self, image):
        syms, lens, _, _ = parse_rl_bwt(image)
        self.bwt = np.repeat(syms, lens.astype(np.int64))
        n = self.n = self.bwt.size
        self.sep = int(syms[lens > 0].min())
        self.N = int((self.bwt == self.sep).sum())
        lf = np.empty(n, np.int64)
        lf[np.argsort(self.bwt, kind="stable")] = np.arange(n)
        # walk every string at once: step t visits the row at position L_k - t of string k
        seen_rows, seen_k, seen_t = [], [], []
        cur, ks, t = np.arange(self.N), np.arange(self.N), 0
        L = np.zeros(self.N, np.int64)
        while cur.size:
            seen_rows.append(cur)
            seen_k.append(ks)
            seen_t.append(np.full(cur.size, t))
            go = self.bwt[cur] != self.sep
            L[ks[~go]] = t
            cur, ks, t = lf[cur[go]], ks[go], t + 1
            if t > n:
                raise ValueError("an LF walk longer than n")
        rows = np.concatenate(seen_rows) if seen_rows else np.zeros(0, np.int64)
        k = np.concatenate(seen_k) if seen_k else np.zeros(0, np.int64)
        tt = np.concatenate(seen_t) if seen_t else np.zeros(0, np.int64)
        if rows.size != n or np.unique(rows).size != n:
            raise ValueError("the strings do not cover the BWT")
        self.k = np.empty(n, np.int64)
        self.p = np.empty(n, np.int64)
        self.k[rows] = k
        self.p[rows] = L[k] - tt
        self.L = L

    def irreducible(self):
        """rows j >= N whose symbol is the separator or differs from row j - 1's"""
        j = np.arange(self.n)
        prev = np.concatenate(([self.bwt[0]], self.bwt[:-1])) if self.n else self.bwt
        return (j >= self.N) & ((self.bwt == self.sep) | (self.bwt != prev))


def lce(arr, sep, x, y, block=64, chunk=1 << 16):
    """cells shared by arr[x ..] and arr[y ..] (vectors of positions), a separator never matching; arr ends with a separator"""
    if x.size > chunk:
        return np.concatenate([lce(arr, sep, x[a:a + chunk], y[a:a + chunk], block, chunk) for a in range(0, x.size, chunk)])
    pad = np.concatenate((arr, np.full(block, sep, arr.dtype)))
    out = np.zeros(x.size, np.int64)
    act = np.arange(x.size)
    off = np.arange(block)
    while act.size:
        a = pad[x[act, None] + out[act, None] + off]
        b = pad[y[act, None] + out[act, None] + off]
        stop = (a != b) | (a == sep)
        hit = stop.any(axis=1)
        first = np.argmax(stop, axis=1)
        out[act[hit]] += first[hit]
        out[act[~hit]] += block
        act = act[~hit]
    return out


def positions(arr, rows):
    """position in arr of every row's suffix: string k starts at the k-th string of arr"""
    t = Text(arr)
    if t.ends.size != rows.N or not np.array_equal(t.ends - t.starts, rows.L):
        raise ValueError("the image is not the collection's")
    return t.starts[rows.k] + rows.p


def lcp_of(arr, image, only=None):
    """(LCP array, Rows, positions); with `only` (a boolean mask of rows) the other entries are left 0"""
    rows = Rows(image)
    pos = positions(arr, rows)
    lcp = np.zeros(rows.n, np.int64)
    j = np.arange(1, rows.n)
    if only is not None:
        j = j[only(rows)[1:]]
    if j.size:
        lcp[j] = lce(arr, rows.sep, pos[j - 1], pos[j])
    return lcp, rows, pos


def check_order(arr, lcp, pos, sep):
    """the first LCP[j] cells of rows j - 1 and j agree and the next cells are ordered, or one of them is a separator"""
    if pos.size < 2:
        return
    x, y, l = pos[:-1], pos[1:], lcp[1:]
    assert np.array_equal(lce(arr, sep, x, y), l)
    a, b = arr[x + l], arr[y + l]
    assert ((a < b) | (a == sep) | (b == sep)).all()
