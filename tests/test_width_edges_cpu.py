"""CPU suite: the construction's width switches through relabelled collections (tests/width_edges.py), without a device.

- The relabelling rule itself, against the oracle run on the relabelled collection, at the edge between 32- and 64-bit level
  symbols (A + nE + 8 = 2^32 - 1 and 2^32) and at A + 1 = 2^32.
- The host induction on the mapped levels: the multi-threaded 32-bit path (ind_phase_mt.hpp) at the narrow edge, the sequential
  64-bit path (ind_phase.hpp) for symbols near 2^63.
- The host tools reverse_bwt and fm_query on .rl_bwt images with 5- and 8-byte symbols below 2^32."""
import subprocess

import numpy as np
import pytest

import grlbwt_b200 as G
from fm_oracle import Text, lib, parse_output, patterns_file, run_tool
from oracle import oracle as O
from width_edges import Base

LEVEL_KEYS = ("pre_sym", "pre_len", "has_hocc", "rule_l", "rule_r", "parse", "str_ptrs", "dict_syms", "dict_len", "dict_freq", "dict_meta")


@pytest.fixture(scope="module")
def base(all_cases):
    return Base(all_cases["u32_small_sigma"])


def edges(b):
    """relabelled alphabets at the narrow / wide switch and at A + 1 = 2^32"""
    return {"narrow": (1 << 32) - 9 - b.nE, "wide": (1 << 32) - 8 - b.nE, "A+1=2^32": (1 << 32) - 1}


@pytest.mark.parametrize("edge", ["narrow", "wide", "A+1=2^32"])
def test_relabelled_levels_match_the_oracle(base, edge):
    m = base.shifted_to_A(edges(base)[edge])
    assert m.wide == (edge != "narrow")
    arr = m.text(np.uint32)
    o = O.Oracle(arr)
    assert o.par_phase() == base.R
    assert o.scalar(0, O.ALPHABET) == m.A and o.scalar(0, O.SUM_LEN) == base.nE
    for lv in range(base.R):
        want = m.level(lv)
        for k, w in zip(LEVEL_KEYS, (O.A_PRE_SYM, O.A_PRE_LEN, O.A_HAS_HOCC, O.A_RULE_L, O.A_RULE_R, O.A_PARSE, O.A_STR_PTRS, O.A_DICT_SYMS,
                                     O.A_DICT_LEN, O.A_DICT_FREQ, O.A_DICT_META)):
            assert np.array_equal(o.array(lv, w).astype(np.uint64), want[k].astype(np.uint64)), (edge, lv + 1, k)
    syms, lens, sb, fb = o.ind_phase()
    ws, wl = m.bwt()
    assert np.array_equal(syms, ws) and np.array_equal(lens, wl) and (sb, fb) == (m.sb, base.fb)
    o.close()


def test_host_induction_on_mapped_levels(all_cases):
    """ind_phase_mt.hpp (threads > 0, 32-bit values) at the narrow edge; ind_phase.hpp (threads = 0) with symbols near 2^63"""
    for name in ("u32_small_sigma", "dna_500", "fuzz_9"):
        b = Base(all_cases[name])
        fp = b.levels[-1]["parse"]
        narrow = b.shifted_to_A((1 << 32) - 9 - b.nE)
        assert not narrow.wide and int(max(L["rule_l"].max(initial=0) for L in narrow.levels())) < 1 << 32
        for threads in (1, 4):
            syms, lens = G.selftest_induce(narrow.levels(), fp, threads)
            ws, wl = narrow.bwt()
            assert np.array_equal(syms, ws) and np.array_equal(lens, wl), (name, threads)
        for A in ((1 << 63) - 1, 1 << 63, (1 << 64) - b.nE - 8):
            m = b.shifted_to_A(A)
            syms, lens = G.selftest_induce(m.levels(), fp, 0)
            ws, wl = m.bwt()
            assert np.array_equal(syms, ws) and np.array_equal(lens, wl), (name, A)


@pytest.mark.parametrize("sb", [5, 8])
def test_host_tools_on_wide_records(all_cases, tmp_path, sb):
    """symbols below 2^32 in 5- and 8-byte records: reverse_bwt gives the text back, fm_query counts as a naive find"""
    for name in ("u32_small_sigma", "u16_small_sigma", "dna_500"):
        arr = all_cases[name]
        b = Base(arr)
        rl = tmp_path / "x.rl_bwt"
        rl.write_bytes(O.rl_bwt_bytes(b.syms, b.lens, sb, b.fb))
        w = arr.dtype.itemsize
        out = tmp_path / "rev.bin"
        r = subprocess.run([lib("reverse_bwt"), str(rl), str(out), "-a", str(w)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert np.array_equal(np.fromfile(out, arr.dtype), arr), name
        t = Text(arr)
        pats = t.patterns(np.random.default_rng(sb))
        pp = tmp_path / "p.bin"
        patterns_file(pp, pats, t.sep, w)
        counts = parse_output(run_tool(lib("fm_query"), rl, pp, w, False))
        assert [c for c, _ in counts] == [len(t.occurrences(p)) for p in pats], name
