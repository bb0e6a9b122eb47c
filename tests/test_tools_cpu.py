"""CPU suite: the .rl_bwt consumer tools (grl2plain, grlbwt2rle, reverse_bwt, bwt_stats, split_runs) -- SURVEY.md 8(f)-4.
Round trip text -> BWT (oracle) -> .rl_bwt -> reverse_bwt == text; parity with the reference's own scripts that build
without SDSL, through their outputs stored in tests/golden/tools_golden.json."""
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import grlbwt_b200 as G
from oracle import oracle as O

NAMES = ["mississippi", "with_empty", "only_empty", "dna_500", "ac_short_3000", "high_bytes", "homopolymer", "u16_small_sigma", "u32_small_sigma",
         "fuzz_5", "fuzz_19", "fuzz_60"]


def tool(name):
    return os.path.join(G.LIB_DIR, name)


@pytest.mark.parametrize("name", NAMES)
def test_tools_round_trip(all_cases, tmp_path, name):
    arr = all_cases[name]
    o = O.Oracle(arr)
    o.par_phase()
    syms, lens, sb, fb = o.ind_phase()
    rl = tmp_path / "x.rl_bwt"
    rl.write_bytes(O.rl_bwt_bytes(syms, lens, sb, fb))
    w = arr.dtype.itemsize
    # reverse_bwt: the original collection, string by string
    out = tmp_path / "rev.bin"
    r = subprocess.run([tool("reverse_bwt"), str(rl), str(out), "-a", str(w)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(np.fromfile(out, arr.dtype), arr)
    # first two strings only
    n_str = int((arr == arr[-1]).sum())
    if n_str >= 2:
        r = subprocess.run([tool("reverse_bwt"), str(rl), str(out), "2", "-a", str(w)], capture_output=True, text=True)
        got = np.fromfile(out, arr.dtype)
        ends = np.flatnonzero(arr == arr[-1])
        assert np.array_equal(got, arr[: ends[1] + 1])
    # grl2plain: the expanded BWT
    plain = tmp_path / "plain.bin"
    r = subprocess.run([tool("grl2plain"), str(rl), str(plain)], capture_output=True, text=True)
    assert r.returncode == 0
    cell = {1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}[1 if sb <= 1 else 2 if sb <= 2 else 4 if sb <= 4 else 8]
    assert np.array_equal(np.fromfile(plain, cell).astype(np.uint64), np.repeat(syms, lens.astype(np.int64)))
    # bwt_stats
    r = subprocess.run([tool("bwt_stats"), str(rl)], capture_output=True, text=True)
    assert f"BWT size (n):            {arr.size}" in r.stdout and f"Number of runs (r):      {len(syms)}" in r.stdout
    assert f"Number of strings:       {n_str}" in r.stdout
    if w == 1:
        pre = tmp_path / "rle"
        r = subprocess.run([tool("grlbwt2rle"), str(rl), str(pre)], capture_output=True, text=True)
        assert r.returncode == 0
        assert np.array_equal(np.fromfile(str(pre) + ".syms", np.uint8).astype(np.uint64), syms)
        assert np.array_equal(np.fromfile(str(pre) + ".len", np.uint32).astype(np.uint64), lens)


def test_bwt_check_accepts_reference_bwts_and_rejects_corrupted(all_cases, tmp_path):
    for name in ("dna_500", "with_empty", "u16_small_sigma", "test_byte_alphabet"):
        arr = all_cases[name]
        o = O.Oracle(arr)
        o.par_phase()
        syms, lens, sb, fb = o.ind_phase()
        txt, rl = tmp_path / "t.bin", tmp_path / "t.rl_bwt"
        arr.tofile(txt)
        rl.write_bytes(O.rl_bwt_bytes(syms, lens, sb, fb))
        w = str(arr.dtype.itemsize)
        r = subprocess.run([tool("bwt_check"), str(txt), str(rl), "-a", w, "-k", "50"], capture_output=True, text=True)
        assert r.returncode == 0 and r.stdout.startswith("OK"), (name, r.stdout)
        if len(syms) > 8:
            bad_s, bad_l = syms.copy(), lens.copy()
            i = len(syms) // 2
            bad_s[[i, i + 1]] = bad_s[[i + 1, i]]          # two runs swapped: totals and maximality still hold
            bad_l[[i, i + 1]] = bad_l[[i + 1, i]]
            rl.write_bytes(O.rl_bwt_bytes(bad_s, bad_l, sb, fb))
            r = subprocess.run([tool("bwt_check"), str(txt), str(rl), "-a", w, "-k", "100000"], capture_output=True, text=True)
            assert r.returncode == 1 and "FAILED" in r.stdout, (name, r.stdout)


def test_truncated_rl_bwt_is_rejected(tmp_path, all_cases):
    """a file that does not hold a whole number of records is an error for every consumer, not a silently shorter BWT"""
    arr = all_cases["dna_500"]
    o = O.Oracle(arr)
    o.par_phase()
    syms, lens, sb, fb = o.ind_phase()
    raw = O.rl_bwt_bytes(syms, lens, sb, fb)
    rl, txt = tmp_path / "cut.rl_bwt", tmp_path / "t.bin"
    arr.tofile(txt)
    rl.write_bytes(raw[:-1])
    for cmd in ([tool("reverse_bwt"), str(rl), str(tmp_path / "o")], [tool("grl2plain"), str(rl), str(tmp_path / "o")],
                [tool("bwt_check"), str(txt), str(rl)], [tool("bwt_stats"), str(rl)], [tool("grlbwt2rle"), str(rl), str(tmp_path / "p")],
                [tool("split_runs"), str(rl), "4", "100", str(tmp_path / "s")]):
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 1 and "truncated" in r.stderr, (cmd[0], r.returncode, r.stderr[-200:])


def test_tools_usage_messages():
    for t in ("grl2plain", "grlbwt2rle", "reverse_bwt", "bwt_stats", "bwt_check", "split_runs"):
        r = subprocess.run([tool(t)], capture_output=True, text=True)
        assert r.returncode == 0 and "usage:" in r.stdout


@pytest.mark.parametrize("sb,fb", [(1, 1), (1, 4), (2, 2), (3, 4), (4, 5), (8, 8), (1, 8), (5, 3)])
def test_rl_bwt_writer_matches_the_format(tmp_path, sb, fb):
    """the host's .rl_bwt writer (two 8-byte stores per record into a slack buffer) == the byte-by-byte definition"""
    import ctypes as C
    from grlbwt_b200.api import lib_host
    rng = np.random.default_rng(sb * 10 + fb)
    L = lib_host()
    L.grlbwt_selftest_write.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int]
    for n in (0, 1, 7, 100003, (1 << 24) // (sb + fb) + 5):   # the last size crosses the writer's flush boundary
        syms = rng.integers(0, 1 << min(8 * sb, 63), size=n, dtype=np.uint64)
        lens = rng.integers(1, 1 << min(8 * fb, 63), size=n, dtype=np.uint64)
        for narrow in ((0, 1) if sb <= 4 else (0,)):
            path = tmp_path / f"w_{sb}_{fb}_{n}_{narrow}.rl_bwt"
            rc = L.grlbwt_selftest_write(str(path).encode(), syms.ctypes.data, lens.ctypes.data, n, sb, fb, narrow)
            assert rc == 0
            assert path.read_bytes() == O.rl_bwt_bytes(syms, lens, sb, fb), (n, narrow)
    # the in-memory packer of grlbwt_build_packed (host induction) produces the same image
    L.grlbwt_selftest_pack.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int]
    for n in (0, 1, 100003):
        syms = rng.integers(0, 1 << min(8 * sb, 32), size=n, dtype=np.uint64)
        lens = rng.integers(1, 1 << min(8 * fb, 32), size=n, dtype=np.uint64)
        img = np.full(16 + n * (sb + fb) + 8, 0xAB, np.uint8)
        for narrow in (0, 1):
            assert L.grlbwt_selftest_pack(img.ctypes.data, img.size - 8, syms.ctypes.data, lens.ctypes.data, n, sb, fb, narrow) == 0
            assert img[:-8].tobytes() == O.rl_bwt_bytes(syms, lens, sb, fb), (n, narrow)
            assert (img[-8:] == 0xAB).all()   # nothing written past the image
        assert L.grlbwt_selftest_pack(img.ctypes.data, 15, syms.ctypes.data, lens.ctypes.data, n, sb, fb, 0) != 0


# ---------------------------------------------------------------- parity with the reference's scripts
# what the reference's scripts produce on these files, stored by tests/golden/make_tools_golden.py
with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tools_golden.json")) as _f:
    REF_OUT = json.load(_f)["cases"]


def sha256_file(path):
    return hashlib.sha256(open(path, "rb").read()).hexdigest()


def _bwt_file(all_cases, tmp_path, name):
    arr = all_cases[name]
    o = O.Oracle(arr)
    o.par_phase()
    syms, lens, sb, fb = o.ind_phase()
    o.close()
    rl = tmp_path / f"{name}.rl_bwt"
    rl.write_bytes(O.rl_bwt_bytes(syms, lens, sb, fb))
    assert sha256_file(rl) == REF_OUT[name]["rl_bwt_sha256"], name
    return rl, syms, lens, sb, fb


def _records(raw):
    sb, fb = int.from_bytes(raw[:8], "little"), int.from_bytes(raw[8:16], "little")
    rec = np.frombuffer(raw[16:], np.uint8).reshape(-1, sb + fb)
    sym = sum(rec[:, i].astype(np.uint64) << np.uint64(8 * i) for i in range(sb))
    ln = sum(rec[:, sb + i].astype(np.uint64) << np.uint64(8 * i) for i in range(fb))
    return sb, fb, np.asarray(sym, np.uint64), np.asarray(ln, np.uint64)


@pytest.mark.parametrize("name", ["rep_50x200k", "mixed_reads", "homopolymers_multi", "test_byte_alphabet"])
def test_tools_match_the_reference_scripts(all_cases, tmp_path, name):
    """grl2plain and grlbwt2rle: the same bytes as scripts/grl2plain.cpp / grlbwt2rle.cpp; bwt_stats: the same report"""
    rl, syms, lens, sb, fb = _bwt_file(all_cases, tmp_path, name)
    want = REF_OUT[name]
    for ours, outs in (("grl2plain", {"{}": "grl2plain_sha256"}), ("grlbwt2rle", {"{}.syms": "grlbwt2rle_syms_sha256", "{}.len": "grlbwt2rle_len_sha256"})):
        b = tmp_path / ("our_" + ours)
        r2 = subprocess.run([tool(ours), str(rl), str(b)], capture_output=True, text=True)
        assert r2.returncode == 0, r2.stderr
        for o_, key in outs.items():
            assert sha256_file(o_.format(b)) == want[key], (ours, o_)
    if len(syms) >= 20:   # (the reference reads one past its sorted lengths when there are fewer than 10 runs)
        r2 = subprocess.run([tool("bwt_stats"), str(rl)], capture_output=True, text=True)
        report = want["bwt_stats_report"]
        assert r2.stdout.splitlines()[: len(report)] == report


@pytest.mark.parametrize("name", ["rep_50x200k", "homopolymers_multi", "mixed_reads"])
def test_split_runs(all_cases, tmp_path, name):
    """split_runs: no run longer than 2^bits - 1, no run across a multiple of n, the same BWT; the reference's output minus the
    zero-length records it emits when a run ends exactly on a block boundary is the same byte stream"""
    rl, syms, lens, sb, fb = _bwt_file(all_cases, tmp_path, name)
    n_syms = int(lens.sum())
    for bits, n in ((3, 1000), (2, 64), (8, 4096), (5, 999983), (12, 0), (4, n_syms + 1)):
        out = tmp_path / f"s_{bits}_{n}"
        r = subprocess.run([tool("split_runs"), str(rl), str(bits), str(n), str(out)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        osb, ofb, s2, l2 = _records(out.read_bytes())
        assert (osb, ofb) == (sb, (bits + 7) // 8)
        assert l2.min() >= 1 and l2.max() <= (1 << bits) - 1
        assert np.array_equal(np.repeat(s2, l2.astype(np.int64)), np.repeat(syms, lens.astype(np.int64)))
        ends = np.cumsum(l2)
        starts = ends - l2
        if n:
            assert ((starts // np.uint64(n)) == ((ends - np.uint64(1)) // np.uint64(n))).all()   # no run crosses a block boundary
            per_block = np.bincount((starts // np.uint64(n)).astype(np.int64))
            dist = np.loadtxt(str(out) + ".dist", skiprows=1, ndmin=2)
            assert dist[:, 1].sum() == per_block.size == -(-n_syms // n)
            assert np.array_equal(np.bincount(per_block, minlength=dist.shape[0])[: dist.shape[0]], dist[:, 1].astype(np.int64))
        if n and n >= 64:   # the reference: asserts (or worse) on tiny blocks and on n = 0
            ref = REF_OUT[name]["split_runs"][f"{bits}_{n}"]
            assert sha256_file(out) == ref["sha256"] and sha256_file(str(out) + ".dist") == ref["dist_sha256"], (bits, n)


def test_parse_rl_bwt_helper(tmp_path):
    """grlbwt_b200.parse_rl_bwt: file path, bytes and uint8 images; malformed images are errors"""
    rng = np.random.default_rng(3)
    for sb, fb in ((1, 1), (1, 4), (3, 4), (8, 8)):
        syms = rng.integers(0, 1 << min(8 * sb, 63), size=1000, dtype=np.uint64)
        lens = rng.integers(1, 1 << min(8 * fb, 63), size=1000, dtype=np.uint64)
        raw = O.rl_bwt_bytes(syms, lens, sb, fb)
        path = tmp_path / "p.rl_bwt"
        path.write_bytes(raw)
        for src in (str(path), raw, np.frombuffer(raw, np.uint8)):
            s2, l2, sb2, fb2 = G.parse_rl_bwt(src)
            assert (sb2, fb2) == (sb, fb) and np.array_equal(s2, syms) and np.array_equal(l2, lens)
        with pytest.raises(ValueError):
            G.parse_rl_bwt(raw[:-1])
    with pytest.raises(ValueError):
        G.parse_rl_bwt(b"\0" * 8)
    with pytest.raises(ValueError):
        G.parse_rl_bwt((9).to_bytes(8, "little") + (1).to_bytes(8, "little"))
