"""GPU suite (-m gpu): the construction at the width limits of its symbols, sort keys, phrase lengths and records.

The inputs are golden cases relabelled by an order-preserving map (tests/width_edges.py), so the expected outputs follow exactly
from the base case's oracle outputs. The shifts land on the switches of the device path:
- 32- or 64-bit level symbols (A + nE + 8 against 2^32, grlgpu.cu level_is_wide, mg2.cuh) and with them device or host induction;
- the symbols per 64-bit suffix sort key (sym_bits = bit_width(A + 1), K = 64 / sym_bits) at K changes and at sym_bits = 64;
- 5- and 8-byte symbols in the header of the .rl_bwt;
- symbols at the top of the u64 range, and the inputs whose arithmetic cannot be represented (refused with GRLGPU_ERR_LIMIT).
Then: phrases of 2^24 cells (the saturated length of the phrase table), every record width of the packed image, and the
device primitives at the types they are called with."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import gen
import grlbwt_b200 as G
from oracle import oracle as O
from width_edges import Base, spread

pytestmark = pytest.mark.gpu
ERR_STATE, ERR_LIMIT = -5, -6
BASES = ("u32_small_sigma", "u16_small_sigma", "dna_500", "mutated_200x5k", "fuzz_9")
TOP64 = (1 << 64) - 1


@pytest.fixture(scope="module")
def bases(all_cases):
    return {name: Base(all_cases[name]) for name in BASES}


def targets(b):
    """(label, cell dtype, relabelling) for one base case"""
    out = []
    for A in ((1 << 16) - 2, (1 << 16) - 1, 1 << 16):                      # A + 1 = 2^16 - 1, 2^16; max_sym = 65535
        out.append((f"u16 A={A}", np.uint16, A))
    for A in ((1 << 32) - 9 - b.nE, (1 << 32) - 8 - b.nE,                  # A + nE + 8 = 2^32 - 1 (narrow), 2^32 (wide)
              (1 << 21) - 2, (1 << 21) - 1, (1 << 22) - 2, (1 << 22) - 1,  # A + 1 = 2^k - 1, 2^k: K = 3 / 2 and 2 / 2
              (1 << 32) - 2, (1 << 32) - 1, 1 << 32):                      # A + 1 = 2^32 - 1, 2^32; max_sym = 2^32 - 1 (sb = 5)
        out.append((f"u32 A={A}", np.uint32, A))
    for A in ((1 << 32) - 1, (1 << 33) - 1, (1 << 63) - 2, (1 << 63) - 1,  # A + 1 = 2^32, 2^33, 2^63 - 1, 2^63
              (1 << 64) - b.nE - 8):                                       # max_sym = 2^64 - nE - 9: the largest accepted
        out.append((f"u64 A={A}", np.uint64, A))
    cases = [(lab, dt, b.shifted_to_A(A)) for lab, dt, A in out if A >= b.A]
    for dt, top, seed in ((np.uint16, (1 << 16) - 1, 1), (np.uint32, (1 << 32) - 1, 2), (np.uint64, (1 << 64) - b.nE - 9, 3)):
        if b.A <= top:
            cases.append((f"{np.dtype(dt).name} sparse", dt, b.mapping(spread(b, top, seed))))
    return cases


def check_rounds(tag, m, arr, flags=0):
    """per round through GrlGpu: mapped round-1 level and dictionary, identical later levels, parse and str_ptrs"""
    b = m.base
    with G.GrlGpu(0, flags | G.FLAG_KEEP_DICT) as ctx:
        ctx.set_text(arr)
        st = ctx.stats()
        assert (st.max_sym, st.sep_sym, st.n_strings) == (m.max_sym, b.sep, len(b.levels[0]["str_ptrs"]) - 1), tag
        for lv in range(b.R):
            r = ctx.round()
            want = m.level(lv)
            t = f"{tag} round {lv + 1}"
            assert r.alphabet == want["alphabet"] and r.tot_phrases == want["tot"], t
            assert r.sym_bytes == (8 if lv == 0 and m.wide else 4), t
            assert r.parse_len == b.levels[lv]["parse_len"] and r.n_phrases == b.levels[lv]["n_phrases"], t
            syms, lens, freqs, metas = ctx.fetch_dictionary()
            for k, got in (("dict_syms", syms), ("dict_len", lens), ("dict_freq", freqs), ("dict_meta", metas)):
                assert np.array_equal(got, want[k]), (t, k)
            L = ctx.fetch_level()
            for k in ("pre_sym", "pre_len", "has_hocc", "rule_l", "rule_r"):
                assert np.array_equal(L[k].astype(np.uint64), want[k].astype(np.uint64)), (t, k)
            assert np.array_equal(ctx.fetch_parse().astype(np.uint64), want["parse"]), (t, "parse")
            assert np.array_equal(ctx.fetch_str_ptrs(), want["str_ptrs"]), (t, "str_ptrs")
        assert r.done, tag


def check_builds(tag, m, arr):
    """the whole .rl_bwt with the device induction (narrow levels), the host induction, and three local ranks"""
    want = m.image(arr.dtype.itemsize)
    img = np.zeros(len(want) + 64, np.uint8)
    for how in ("default", "host", "3 ranks"):
        if how == "host":
            os.environ["GRLBWT_HOST_INDUCTION"] = "1"
        try:
            nb, n_runs, sb, fb, info = G.build_bwt_packed(arr, img, devices=[0, 0, 0] if how == "3 ranks" else [0], n_threads=4)
        finally:
            os.environ.pop("GRLBWT_HOST_INDUCTION", None)
        assert img[:nb].tobytes() == want, (tag, how)
        if how == "default":
            assert bool(info["induced_on_device"]) == (not m.wide), (tag, info)
        if how == "host":
            assert not info["induced_on_device"], tag


def check_fm(tag, m, arr, ctx):
    """below 2^32: the inversion returns the relabelled text, and relabelled patterns count as the base's patterns"""
    if m.max_sym >= 1 << 32:
        return
    img = m.image(arr.dtype.itemsize)
    got, _ = ctx.invert(img, arr.dtype.itemsize)
    assert np.array_equal(got, arr), (tag, "invert")
    b = m.base
    rng = np.random.default_rng(7)
    pats = []
    ends = np.flatnonzero(b.arr == b.sep)
    starts = np.concatenate(([0], ends[:-1] + 1))
    for _ in range(64):
        k = int(rng.integers(0, ends.size))
        if ends[k] == starts[k]:
            continue
        p = int(rng.integers(starts[k], ends[k]))
        pats.append(b.arr[p: min(ends[k], p + int(rng.integers(1, 9)))].astype(np.uint64))
    pats += [b.alpha[i: i + 1] for i in range(min(b.alpha.size, 8))]
    base_img = O.rl_bwt_bytes(b.syms, b.lens, b.sb, b.fb)
    ctx.fm_load(base_img)
    sp0, ep0, _ = ctx.fm_count([p.astype(b.arr.dtype) for p in pats])
    ctx.fm_load(img)
    sp1, ep1, _ = ctx.fm_count([m.g(p).astype(arr.dtype) for p in pats])
    assert np.array_equal(ep1 - sp1, ep0 - sp0), (tag, "fm_count")
    ctx.fm_drop()


@pytest.mark.parametrize("name", BASES)
def test_relabelled_at_width_switches(bases, name):
    b = bases[name]
    with G.GrlGpu(0) as fm_ctx:
        for tag, dt, m in targets(b):
            tag = f"{name} {tag}"
            arr = m.text(dt)
            assert int(arr.max()) == m.max_sym
            check_rounds(tag, m, arr)
            check_builds(tag, m, arr)
            check_fm(tag, m, arr, fm_ctx)


def test_relabelled_dedup_and_refinement_paths(bases):
    """the uncached dedup and the refinement by prefix doubling at the wide edge and with sym_bits = 64"""
    b = bases["mutated_200x5k"]
    for A in ((1 << 32) - 8 - b.nE, (1 << 64) - b.nE - 8):
        m = b.shifted_to_A(A)
        arr = m.text(np.uint64)
        for flags in (G.FLAG_FORCE_UNCACHED, G.FLAG_FORCE_DOUBLING):
            check_rounds(f"A={A} flags={flags}", m, arr, flags)


# ------------------------------------------------------------------ inputs the arithmetic cannot represent
def test_symbols_too_close_to_2_64_are_refused(bases, tmp_path):
    """max_sym = 2^64 - 1 (A wraps), 2^64 - 2 (A + 1 wraps) and 2^64 - nE - 8 (A + nE + 8 > 2^64): GRLGPU_ERR_LIMIT from the library,
    the Python API and the CLI, on one rank and on three; max_sym = 2^64 - nE - 9 is built (test_relabelled_at_width_switches)"""
    b = bases["u32_small_sigma"]
    for max_sym in ((1 << 64) - b.nE - 8, (1 << 64) - 2, (1 << 64) - 1):
        m = b.shifted_to_A(max_sym + 1)
        arr = m.text(np.uint64)
        assert int(arr.max()) == max_sym
        with G.GrlGpu(0) as ctx:
            ctx.set_text(arr)
            if max_sym == TOP64:
                with pytest.raises(G.GrlGpuError) as e:
                    ctx.stats()
            else:
                assert ctx.stats().max_sym == max_sym
                with pytest.raises(G.GrlGpuError) as e:
                    ctx.round()
            assert e.value.status == ERR_LIMIT, max_sym
        for devices in ([0], [0, 0, 0]):
            with pytest.raises(G.GrlGpuError) as e:
                G.build_bwt_packed(arr, np.zeros(16 + arr.size * 16, np.uint8), devices=devices, n_threads=2)
            assert e.value.status == ERR_LIMIT, (max_sym, devices, str(e.value))
        with pytest.raises(G.GrlGpuError) as e:
            G.build_bwt(arr)
        assert e.value.status == ERR_LIMIT
        inp = tmp_path / "top.bin"
        arr.tofile(inp)
        r = subprocess.run([os.path.join(G.LIB_DIR, "grlbwt"), str(inp), "-a", "8", "-T", str(tmp_path)], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 1 and "size limit of the device path exceeded" in r.stderr and "2^64" in r.stderr, (max_sym, r.stdout, r.stderr)
        assert not (tmp_path / "top.rl_bwt").exists()


# ------------------------------------------------------------------ phrases of 2^24 cells
def long_phrases():
    """strings C..CA..A (no LMS position: one phrase each) of 2^24 + {-3 .. 1} cells, each twice, and a pair that shares its first
    2^24 + 1 cells and differs only in length (the hash key holds a saturated length; only the bitmaps tell the two apart)"""
    T, parts = 1 << 24, []
    for d in (-3, -2, -1, 0, 1):
        n = T + d
        s = np.full(n + 1, ord("A"), np.uint8)
        s[: n // 2] = ord("C")
        s[-1] = 10
        parts += [s, s]
    for n in (T + 1, T + 2):
        s = np.full(n + 1, ord("A"), np.uint8)
        s[:1000] = ord("C")
        s[-1] = 10
        parts.append(s)
    return np.concatenate(parts)


def test_phrases_of_2_24_cells():
    """every string is one phrase (its cells and the separator). The oracle takes too long at this size, so the rounds are checked
    against the dictionary the strings imply (in the oracle's order, as on a 2^12 analog of the collection), the two dedup paths against
    each other, and the .rl_bwt by inverting it"""
    T, arr = 1 << 24, long_phrases()
    want_len = np.array([T + 2, T + 3, T - 2, T - 1, T, T + 1, T + 2], np.uint64)   # the pair first: its strings have the fewest C
    want_freq = np.array([1, 1, 2, 2, 2, 2, 2], np.uint64)
    got = []
    for flags in (0, G.FLAG_FORCE_UNCACHED):
        with G.GrlGpu(0, flags | G.FLAG_KEEP_DICT) as ctx:
            ctx.set_text(arr)
            ctx.stats()
            r = ctx.round()
            assert r.done and (r.n_phrases, r.dict_syms, r.parse_len) == (7, int(want_len.sum()), 12), flags
            syms, lens, freqs, metas = ctx.fetch_dictionary()
            assert np.array_equal(lens, want_len) and np.array_equal(freqs, want_freq), (flags, lens, freqs)
            parse = ctx.fetch_parse().astype(np.uint64)
            assert np.array_equal(parse, metas[[2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 0, 1]]) and np.unique(metas).size == 7, (flags, parse, metas)
            off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
            assert np.array_equal(syms[off[0]: off[1]], arr[-(2 * T + 5): -(T + 3)]) and np.array_equal(syms[off[1]: off[2]], arr[-(T + 3):]), flags
            L = ctx.fetch_level()
            got.append((syms, lens, freqs, metas, parse, L))
    for a, b in zip(got[0][:5], got[1][:5]):
        assert np.array_equal(a, b)
    for k in ("pre_sym", "pre_len", "has_hocc", "rule_l", "rule_r"):
        assert np.array_equal(got[0][5][k], got[1][5][k]), k
    img = np.zeros(16 + 64 * 1024, np.uint8)
    nb, n_runs, sb, fb, _ = G.build_bwt_packed(arr, img)
    assert (sb, fb) == (1, 4)
    out, _ = G.invert_rl_bwt(img[:nb].tobytes())
    assert np.array_equal(out, arr)
    with pytest.raises(G.GrlGpuError) as e:   # the multi-GPU round keeps no bitmaps at the owner: it refuses such phrases
        G.build_bwt_packed(arr, img, devices=[0, 0], n_threads=2)
    assert e.value.status == ERR_LIMIT


# ------------------------------------------------------------------ record widths of the packed image
def packed_lib():
    L = G.lib_gpu()
    vp, u64 = C.c_void_p, C.c_uint64
    L.grlgpu_keep_level.argtypes = [vp]
    L.grlgpu_induce.argtypes = [vp, vp, u64, C.c_int, u64, C.POINTER(u64)]
    L.grlgpu_fetch_bwt.argtypes = [vp, vp, vp]
    L.grlgpu_fetch_bwt_packed.argtypes = [vp, C.c_int, C.c_int, vp, u64, C.POINTER(u64)]
    return L


def homopolymers():
    parts = [b"A" * 255 + b"\n", b"C" * 256 + b"\n", b"G" * 65535 + b"\n", b"T" * 65536 + b"\n", b"ACGT" * 20 + b"A" * 255 + b"C" * 65536 + b"\n"]
    return np.frombuffer(b"".join(parts), np.uint8).copy()


@pytest.mark.parametrize("case", ["byte", "u16", "homopolymers", "reads_45M"])
def test_packed_record_widths(all_cases, case):
    arr = {"byte": lambda: all_cases["mutated_200x5k"], "u16": lambda: all_cases["u16_rand"], "homopolymers": homopolymers,
           "reads_45M": lambda: gen.dna_reads(320000, 150, seed=9)}[case]()
    L = packed_lib()
    with G.GrlGpu(0) as ctx:
        ctx.set_text(arr)
        while True:
            r = ctx.round()
            assert L.grlgpu_keep_level(ctx._h) == 0
            if r.done:
                break
        n_runs = C.c_uint64()
        assert L.grlgpu_induce(ctx._h, None, r.parse_len, r.cell_bytes_out, arr.size, C.byref(n_runs)) == 0
        n = n_runs.value
        syms, lens = np.zeros(n, np.uint32), np.zeros(n, np.uint32)
        assert L.grlgpu_fetch_bwt(ctx._h, syms.ctypes.data_as(C.c_void_p), lens.ctypes.data_as(C.c_void_p)) == 0
        bs, bl = O.rle(O.bcr_bwt(arr)) if arr.size < 4_000_000 else (None, None)
        if bs is not None:
            assert np.array_equal(syms, bs) and np.array_equal(lens, bl)
        s_need, f_need = (int(syms.max()).bit_length() + 7) // 8, (int(lens.max()).bit_length() + 7) // 8
        # the little-endian bytes of every symbol and length: record (sb, fb) of run i is S[i, :sb] followed by F[i, :fb]
        S, F = syms.astype("<u8").view(np.uint8).reshape(n, 8), lens.astype("<u8").view(np.uint8).reshape(n, 8)
        big = n > 32 << 20   # above the piece size of the packing: records of 3, 5 and 7 bytes cross a piece boundary
        img = np.zeros(16 + n * 16, np.uint8)
        nb = C.c_uint64()
        with G.GrlGpu(0) as ictx:
            for sb in range(1, 9):
                for fb in range(1, 9):
                    rc = L.grlgpu_fetch_bwt_packed(ctx._h, sb, fb, img.ctypes.data_as(C.c_void_p), img.size, C.byref(nb))
                    if sb < s_need or fb < f_need:
                        assert rc == ERR_STATE, (case, sb, fb)
                        continue
                    rec = sb + fb
                    assert rc == 0 and nb.value == 16 + n * rec, (case, sb, fb)
                    assert img[:16].view(np.uint64).tolist() == [sb, fb], (case, sb, fb)
                    body = img[16:16 + n * rec].reshape(n, rec)
                    assert np.array_equal(body[:, :sb], S[:, :sb]) and np.array_equal(body[:, sb:], F[:, :fb]), (case, sb, fb)
                    # the images are read back: every odd record size with the narrowest or the widest symbols (two pairs on the big case)
                    if (rec % 2 and sb in (s_need, 8)) and (not big or (sb, fb) in ((s_need, f_need + 1 - (s_need + f_need) % 2), (8, 7))):
                        want = img[:nb.value].copy()
                        got, _ = ictx.invert(want, arr.dtype.itemsize)
                        assert np.array_equal(got, arr), (case, sb, fb)
                        ictx.fm_load(want)
                        pats = [arr[i: i + 6] for i in (0, 100, 1000) if i + 6 < arr.size and not (arr[i: i + 6] == arr[-1]).any()]
                        if pats:
                            sp, ep, _ = ictx.fm_count(pats)
                            ictx.fm_load(O.rl_bwt_bytes(syms, lens, s_need, f_need))
                            sp0, ep0, _ = ictx.fm_count(pats)
                            assert np.array_equal(ep - sp, ep0 - sp0), (case, sb, fb)
        assert big == (case == "reads_45M"), (case, n)
        # a failed width leaves the context usable
        rc = L.grlgpu_fetch_bwt_packed(ctx._h, s_need, f_need, img.ctypes.data_as(C.c_void_p), img.size, C.byref(nb))
        assert rc == 0 and img[:nb.value].tobytes() == O.rl_bwt_bytes(syms, lens, s_need, f_need)


# ------------------------------------------------------------------ primitives at the types they are called with
SIZES = [1, 8192, 8193, (1 << 21) + 5, 5_000_003]


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("dtype", [np.uint32, np.uint64])
def test_scan_same_type(n, dtype):
    rng = np.random.default_rng(n)
    top = 1 << 31 if dtype == np.uint32 else 1 << 62   # u32 sums wrap mod 2^32
    a = rng.integers(0, top, size=n, dtype=dtype)
    ref = np.cumsum(a, dtype=dtype) - a
    tot = int(a.sum(dtype=dtype))
    for off in (0, 1, 3):
        for in_place in (False, True):
            out, t = G.api.selftest_scan_same(a, off, in_place)
            assert t == tot and np.array_equal(out, ref), (n, off, in_place)


@pytest.mark.parametrize("n", SIZES)
def test_radix_sort_u32(n):
    rng = np.random.default_rng(n + 1)
    for bits in (8, 24, 32):
        keys = rng.integers(0, 1 << 32, size=n, dtype=np.uint64).astype(np.uint32)   # bits above n_bits are carried, not sorted on
        if n > 1000:
            keys[: n // 3] = keys[n // 3: 2 * (n // 3)]
        vals = np.arange(n, dtype=np.uint32)
        k, v = G.api.selftest_sort32(keys, vals, bits)
        order = np.argsort(keys & np.uint32((1 << bits) - 1) if bits < 32 else keys, kind="stable")
        assert np.array_equal(k, keys[order]) and np.array_equal(v, vals[order]), (n, bits)


@pytest.mark.parametrize("n", SIZES)
def test_radix_partition_u32(n):
    rng = np.random.default_rng(n + 2)
    keys = rng.integers(0, 1 << 32, size=n, dtype=np.uint64).astype(np.uint32)
    vals = rng.integers(0, 1 << 32, size=n, dtype=np.uint64).astype(np.uint32)
    for shift in (0, 8, 24):
        k, v = G.api.selftest_sort32(keys, vals, partition_shift=shift)
        order = np.argsort((keys >> np.uint32(shift)) & np.uint32(255), kind="stable")
        assert np.array_equal(k, keys[order]) and np.array_equal(v, vals[order]), (n, shift)


@pytest.mark.parametrize("n", [8193, (1 << 21) + 5])
def test_radix_sort_u64_keys_above_n_bits(n):
    """the 64-bit sort carries bits above n_bits (whole digits) unsorted, stably"""
    rng = np.random.default_rng(n + 3)
    keys = rng.integers(0, 1 << 63, size=n, dtype=np.uint64)
    vals = np.arange(n, dtype=np.uint32)
    for bits in (16, 40):
        k, v = G.selftest_sort(keys, vals, bits)
        order = np.argsort(keys & np.uint64((1 << bits) - 1), kind="stable")
        assert np.array_equal(k, keys[order]) and np.array_equal(v, vals[order]), (n, bits)
