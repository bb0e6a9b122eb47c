"""Order-preserving relabelling of a collection, and what it does to the construction's outputs.

Relabel every symbol but the separator with an increasing map g (the separator stays the smallest symbol). Every symbol
comparison then comes out the same, so the expected outputs follow from those of the base collection:
- the BWT is the relabelled BWT, with the same run lengths;
- every round's parse, str_ptrs, phrase counts, has_hocc and pre_len are identical;
- round 1's level (pre_sym, rule_l, rule_r) maps v -> g(v) for text symbols v < A and v -> v + (A' - A) for the dummies A + 1,
  A + 2 and the metasymbols A + 3 + r (A = max_sym + 1 of the base, A' of the relabelled collection);
- the levels of rounds 2 and on are identical.
nE, the number of round-1 dictionary symbols, does not change, so a shift can be chosen to land exactly on a width switch."""
import numpy as np

from oracle import oracle as O

U64 = np.uint64


class Base:
    """one base collection through the oracle: levels, parses, str_ptrs, dictionary and BWT"""

    def __init__(self, arr):
        self.arr = np.ascontiguousarray(arr)
        o = O.Oracle(self.arr)
        self.R = o.par_phase()
        self.sep = int(self.arr[-1])
        self.A = o.scalar(0, O.ALPHABET)
        self.nE = o.scalar(0, O.SUM_LEN)
        self.levels = []
        for lv in range(self.R):
            self.levels.append({"alphabet": o.scalar(lv, O.ALPHABET), "tot": o.scalar(lv, O.TOT_PHRASES),
                                "rule_l": o.array(lv, O.A_RULE_L), "rule_r": o.array(lv, O.A_RULE_R),
                                "has_hocc": o.array(lv, O.A_HAS_HOCC).astype(np.uint8),
                                "pre_sym": o.array(lv, O.A_PRE_SYM), "pre_len": o.array(lv, O.A_PRE_LEN),
                                "parse": o.array(lv, O.A_PARSE), "str_ptrs": o.array(lv, O.A_STR_PTRS),
                                "dict_syms": o.array(lv, O.A_DICT_SYMS), "dict_len": o.array(lv, O.A_DICT_LEN),
                                "dict_freq": o.array(lv, O.A_DICT_FREQ), "dict_meta": o.array(lv, O.A_DICT_META),
                                "n_phrases": o.scalar(lv, O.D), "parse_len": o.scalar(lv, O.PARSE_LEN)})
        self.syms, self.lens, self.sb, self.fb = o.ind_phase()
        o.close()
        self.alpha = np.unique(self.arr[self.arr != self.sep]).astype(U64)   # the non-separator symbols, ascending

    def mapping(self, new_alpha):
        return Relabel(self, np.asarray(new_alpha, U64))

    def shifted(self, delta):
        return self.mapping(self.alpha + U64(delta))

    def shifted_to_A(self, A_new):
        """the shift that makes the relabelled alphabet (max_sym + 1) equal to A_new"""
        return self.shifted(int(A_new) - self.A)


class Relabel:
    """the base collection under g: alpha[i] -> new_alpha[i], separator fixed"""

    def __init__(self, base, new_alpha):
        assert new_alpha.size == base.alpha.size and (new_alpha[1:] > new_alpha[:-1]).all()
        assert new_alpha.size == 0 or int(new_alpha[0]) > base.sep
        self.base = base
        self.new_alpha = new_alpha
        self.max_sym = int(new_alpha[-1]) if new_alpha.size else base.sep
        self.A = self.max_sym + 1
        self.dA = self.A - base.A

    def g(self, v):
        """text symbols through g, values >= A (dummies, metasymbols) shifted by dA; the separator stays"""
        v = np.asarray(v, U64)
        out = v.copy()
        txt = (v < U64(self.base.A)) & (v != U64(self.base.sep))
        out[txt] = self.new_alpha[np.searchsorted(self.base.alpha, v[txt])]
        hi = v >= U64(self.base.A)
        out[hi] = (v[hi].astype(object) + self.dA).astype(U64)
        return out

    def text(self, dtype):
        a = self.base.arr.astype(U64)
        return self.g(a).astype(dtype)

    def level(self, lv):
        """expected level of round lv + 1 (u64 arrays)"""
        L = self.base.levels[lv]
        out = {k: L[k] for k in ("has_hocc", "pre_len", "parse", "str_ptrs", "dict_len", "dict_freq", "dict_meta", "tot")}
        for k in ("pre_sym", "rule_l", "rule_r", "dict_syms"):
            out[k] = self.g(L[k]) if lv == 0 else L[k]
        out["alphabet"] = self.A if lv == 0 else L["alphabet"]
        return out

    def levels(self):
        return [self.level(lv) for lv in range(self.base.R)]

    @property
    def wide(self):
        """64-bit level symbols in round 1"""
        return self.A + self.base.nE + 8 >= 1 << 32

    @property
    def sb(self):
        """the reference's header rule: symbol bytes of max_sym + 1 + 3"""
        return max(1, (self.max_sym + 4).bit_length() + 7 >> 3)

    def fb(self, cell_bytes):
        """the reference's header rule: length bytes of max_sym_freq, which is the largest symbol count for byte cells and n for
        wider ones (utils.cpp:117,161-175), so a byte case widened to larger cells may need more length bytes"""
        if cell_bytes == 1:
            return self.base.fb
        return max(1, (self.base.arr.size.bit_length() + 7) >> 3)

    def bwt(self):
        return self.g(self.base.syms), self.base.lens

    def image(self, cell_bytes):
        s, l = self.bwt()
        return O.rl_bwt_bytes(s, l, self.sb, self.fb(cell_bytes))


def spread(base, top, seed):
    """a sparse, non-affine increasing map of the base's symbols into (sep, top]: random distinct values"""
    rng = np.random.default_rng(seed)
    m, lo = base.alpha.size, base.sep + 1
    if top - lo + 1 < 4 * m:
        raise ValueError("range too small")
    picks = set()
    while len(picks) < m - 1:
        picks.add(int(rng.integers(lo, top, dtype=np.uint64)))   # below top: top itself is always used, so max_sym = top
    return sorted(picks) + [top]
