"""GPU suite: grlgpu_invert (the .rl_bwt image back to the collection on the device), its Python binding invert_rl_bwt and the
reverse_bwt_gpu tool, against the texts themselves and the host tool reverse_bwt."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import grlbwt_b200 as G
from grlbwt_b200.api import Invert, lib_gpu
from oracle import oracle as O

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_ILL_FORMED, ERR_LIMIT = -1, -2, -6
AUTO, WALK, JUMP = 0, G.FLAG_FORCE_WALK, G.FLAG_FORCE_JUMP


def tool(name):
    return os.path.join(G.LIB_DIR, name)


def oracle_image(arr):
    o = O.Oracle(arr)
    o.par_phase()
    syms, lens, sb, fb = o.ind_phase()
    o.close()
    return O.rl_bwt_bytes(syms, lens, sb, fb), syms


def host_reverse(tmp_path, raw, w, n_seqs=None):
    rl, out = tmp_path / "h.rl_bwt", tmp_path / "h.out"
    rl.write_bytes(raw)
    cmd = [tool("reverse_bwt"), str(rl), str(out)] + ([] if n_seqs is None else [str(n_seqs)]) + ["-a", str(w)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return out.read_bytes()


def lf_of(L):
    """LF of a BWT given as a symbol array: C[c] + rank_c(j), by a stable sort"""
    order = np.argsort(L, kind="stable")
    lf = np.empty(L.size, np.int64)
    lf[order] = np.arange(L.size)
    return lf


def image_of_runs(syms, lens, sb=4, fb=4):
    return O.rl_bwt_bytes(np.asarray(syms, np.uint64), np.asarray(lens, np.uint64), sb, fb)


def test_every_case_on_both_paths(all_cases, tmp_path):
    """every golden case inverts to its text automatically, by the walk and by pointer jumping; a sample also against the bytes
    reverse_bwt writes"""
    sample = {"mississippi", "with_empty", "only_empty", "homopolymers_multi", "u16_small_sigma", "u32_small_sigma", "fuzz_5", "test_2bytes_alphabet"}
    for name, arr in all_cases.items():
        raw, syms = oracle_image(arr)
        w = arr.dtype.itemsize
        if syms.max() >= (1 << 32):   # beyond the device's 32-bit symbols
            with pytest.raises(G.GrlGpuError) as e:
                G.invert_rl_bwt(raw, w)
            assert e.value.status == ERR_LIMIT, name
            continue
        for flags, path in ((AUTO, None), (WALK, 0), (JUMP, 1)):
            got, info = G.invert_rl_bwt(raw, w, flags=flags)
            assert got.tobytes() == arr.tobytes(), (name, flags)
            assert info["n"] == arr.size and info["n_out"] == arr.size and info["n_strings"] == int((arr == arr[-1]).sum()), (name, info)
            assert path is None or info["path"] == path, (name, info)
        if name in sample:
            assert host_reverse(tmp_path, raw, w) == arr.tobytes(), name


@pytest.mark.parametrize("name", ["with_empty", "dna_500", "u16_small_sigma", "fuzz_19", "only_empty"])
def test_first_strings_match_reverse_bwt(all_cases, tmp_path, name):
    arr = all_cases[name]
    raw, _ = oracle_image(arr)
    w = arr.dtype.itemsize
    N = int((arr == arr[-1]).sum())
    for k in sorted({0, 1, 2, max(0, N - 1), N, N + 5}):
        want = host_reverse(tmp_path, raw, w, k)
        for flags in (WALK, JUMP):
            got, info = G.invert_rl_bwt(raw, w, n_seqs=k, flags=flags)
            assert got.tobytes() == want, (name, k, flags)
            assert info["n_out"] * w == len(want)


@pytest.mark.parametrize("name", ["rep_50x200k", "homopolymers_multi", "mixed_reads"])
def test_runs_that_are_not_maximal(all_cases, tmp_path, name):
    """split_runs output (runs cut at a bit limit and at block ends) and zero-length records invert to the same text"""
    arr = all_cases[name]
    raw, _ = oracle_image(arr)
    rl = tmp_path / "in.rl_bwt"
    rl.write_bytes(raw)
    for bits, n in ((3, 1000), (2, 64), (8, 4096), (5, 999983), (12, 0)):
        out = tmp_path / f"s_{bits}_{n}"
        r = subprocess.run([tool("split_runs"), str(rl), str(bits), str(n), str(out)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        for flags in (AUTO, WALK, JUMP):
            got, _ = G.invert_rl_bwt(str(out), 1, flags=flags)
            assert got.tobytes() == arr.tobytes(), (bits, n, flags)
    syms, lens, sb, fb = G.parse_rl_bwt(raw)
    mid = syms.size // 2
    # zero-length records: first (with a symbol below the separator), in the middle, last
    s2 = np.concatenate(([0], syms[:mid], [syms[mid]], syms[mid:], [syms[-1] + 1]))
    l2 = np.concatenate(([0], lens[:mid], [0], lens[mid:], [0]))
    for flags in (AUTO, WALK, JUMP):
        got, _ = G.invert_rl_bwt(image_of_runs(s2, l2, sb, fb), 1, flags=flags)
        assert got.tobytes() == arr.tobytes(), flags


@pytest.mark.parametrize("name,path", [("reads_2M", 0), ("rep_100x1M", 1), ("u16_20M", None), ("mixed_200k", None)])
def test_round_trip_at_scale(name, path):
    """build_bwt_packed, then automatic inversion: the text again; reads take the walk, long strings pointer jumping"""
    import gen
    arr = {"reads_2M": lambda: gen.dna_reads(2000000, 150, seed=42), "rep_100x1M": lambda: gen.repetitive_genomes(100, 1000000, seed=7),
           "u16_20M": lambda: gen.int_alphabet(20000000, np.uint16, 65535, 1000, seed=11),
           "mixed_200k": lambda: gen.mixed_reads(200000, 300, 150, 10000, seed=5)}[name]()
    img = np.empty(16 + arr.size * 16, np.uint8)
    nb, _, _, _, _ = G.build_bwt_packed(arr, img, n_threads=8)
    got, info = G.invert_rl_bwt(img[:nb], arr.dtype.itemsize)
    assert info["n"] == arr.size and got.tobytes() == arr.tobytes(), (name, info)
    assert path is None or info["path"] == path, (name, info)


def test_errors(all_cases):
    arr = all_cases["dna_500"]
    raw, _ = oracle_image(arr)
    for bad in (raw[:-1], raw[:10], raw[:16], (0).to_bytes(8, "little") + raw[8:], (9).to_bytes(8, "little") + raw[8:],
                raw[:8] + (9).to_bytes(8, "little") + raw[16:]):
        with pytest.raises(G.GrlGpuError) as e:
            G.invert_rl_bwt(bad, 1)
        assert e.value.status == ERR_ARG
    # cell width: refused by the binding and by the library itself
    with pytest.raises(G.GrlGpuError) as e:
        G.invert_rl_bwt(raw, 3)
    assert e.value.status == ERR_ARG
    with G.GrlGpu(0) as ctx:
        buf, info = np.zeros(arr.size * 4, np.uint8), Invert()
        img = np.frombuffer(raw, np.uint8)
        for w in (0, 3, 16):
            assert lib_gpu().grlgpu_invert(ctx._h, img.ctypes.data, img.size, w, (1 << 64) - 1, buf.ctypes.data, buf.size, C.byref(info)) == ERR_ARG
    # output buffer too small: the size needed comes back
    with pytest.raises(G.GrlGpuError) as e:
        G.invert_rl_bwt(raw, 1, out=np.zeros(arr.size - 1, np.uint8))
    assert e.value.status == ERR_ARG and e.value.info["n_out"] == arr.size
    ends = np.flatnonzero(arr == arr[-1])
    with pytest.raises(G.GrlGpuError) as e:
        G.invert_rl_bwt(raw, 2, n_seqs=3, out=np.zeros(8, np.uint8))
    assert e.value.status == ERR_ARG and e.value.info["n_out"] == ends[2] + 1
    # a symbol of 2^32 or more
    with pytest.raises(G.GrlGpuError) as e:
        G.invert_rl_bwt(image_of_runs([1, 1 << 32, 2], [1, 1, 1], 5, 1), 8)
    assert e.value.status == ERR_LIMIT
    # run lists that are not a BWT: LF has a cycle without separator row (length 2, where jumping stops moving, and length 3,
    # where it moves at every round)
    for L in (np.array([1, 3, 2]), np.array([1, 4, 2, 3]), np.array([1, 2, 1, 4, 3, 5])):
        lf, sep = lf_of(L), L.min()
        on_cycle = []
        for j in range(L.size):   # rows whose orbit meets no separator row
            k, seen = j, False
            for _ in range(L.size):
                seen |= L[k] == sep
                k = lf[k]
            if not seen:
                on_cycle.append(j)
        assert on_cycle, L
        s, ln = O.rle(L)
        for flags in (WALK, JUMP, AUTO):
            with pytest.raises(G.GrlGpuError) as e:
                G.invert_rl_bwt(image_of_runs(s, ln), 1, flags=flags)
            assert e.value.status == ERR_ILL_FORMED, (L, flags)


def test_context_is_left_untouched(all_cases):
    """inversion on a context between rounds changes neither the rounds nor a later inversion"""
    a, b = all_cases["mutated_200x5k"], all_cases["reads_2000x150"]
    raw, _ = oracle_image(a)
    with G.GrlGpu(0) as ref:
        ref.set_text(b)
        want = []
        while True:
            r = ref.round()
            want.append((ref.fetch_parse().copy(), ref.level_checksum()))
            if r.done:
                break
    with G.GrlGpu(0) as ctx:
        first, _ = ctx.invert(raw)
        ctx.set_text(b)
        got = []
        while True:
            r = ctx.round()
            again, _ = ctx.invert(raw)
            assert again.tobytes() == first.tobytes() == a.tobytes()
            got.append((ctx.fetch_parse().copy(), ctx.level_checksum()))
            if r.done:
                break
        last, _ = ctx.invert(raw)
        assert last.tobytes() == a.tobytes()
    assert len(got) == len(want)
    for (p1, c1), (p2, c2) in zip(got, want):
        assert np.array_equal(p1, p2) and c1 == c2


@pytest.mark.parametrize("name", ["with_empty", "dna_500", "u16_small_sigma", "homopolymers_multi"])
def test_tool_matches_reverse_bwt(all_cases, tmp_path, name):
    arr = all_cases[name]
    raw, _ = oracle_image(arr)
    rl = tmp_path / "x.rl_bwt"
    rl.write_bytes(raw)
    for extra in ([], ["2"], ["-a", "2"], ["3", "-a", "2"]):
        outs = []
        for t in ("reverse_bwt", "reverse_bwt_gpu"):
            out = tmp_path / t
            r = subprocess.run([tool(t), str(rl), str(out)] + extra, capture_output=True, text=True)
            assert r.returncode == 0, r.stderr
            outs.append(out.read_bytes())
        assert outs[0] == outs[1], (name, extra)
    bad = tmp_path / "bad.rl_bwt"
    bad.write_bytes(raw[:-1])
    r = subprocess.run([tool("reverse_bwt_gpu"), str(bad), str(tmp_path / "o")], capture_output=True, text=True)
    assert r.returncode == 1 and "invalid argument" in r.stderr
