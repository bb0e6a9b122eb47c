"""GPU suite: the search with mismatches on the device (grlgpu_fm_approx_count / _locate, GrlGpu.fm_approx_*, fm_query_gpu -k)
against every window of the collections, the exact search and the host tool fm_query -k."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import grlbwt_b200 as G
from approx_oracle import mutate, naive, naive_counts, patterns, pigeonhole
from fm_oracle import Text, image_of, lib, patterns_file
from grlbwt_b200.api import FmApprox, lib_gpu

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_ILL_FORMED, ERR_STATE, ERR_LIMIT = -1, -2, -5, -6
AUTO, WALK, JUMP = 0, G.FLAG_FORCE_WALK, G.FLAG_FORCE_JUMP
K3_CASES = ("mississippi", "dna_500", "u16_small_sigma", "reads_2000x150", "fuzz_0", "test_2bytes_alphabet")


def check_hits(hit_off, sp, ep, mm, want, kmax):
    """per pattern: hits disjoint and ascending, and their rows per d add up to the oracle's occurrences per d (want[q][d])"""
    for q, cnt in enumerate(want):
        a, b = int(hit_off[q]), int(hit_off[q + 1])
        s, e, d = sp[a:b].astype(np.int64), ep[a:b].astype(np.int64), mm[a:b]
        assert (e > s).all() and (s[1:] >= e[:-1]).all(), q
        for x in range(kmax + 1):
            assert int((e - s)[d == x].sum()) == int(cnt[x]), (q, x)


def test_every_case(all_cases):
    """every golden case with 32-bit symbols up to 3 M cells (test_at_scale takes the larger ones), k = 0, 1, 2 (and 3 on a few):
    hits against every window, k = 0 against fm_count, the occurrences against every window on the three locate paths, which
    agree row for row"""
    for name, arr in all_cases.items():
        if arr.size > 3_000_000:   # the naive oracle reads every window once per pattern
            continue
        raw, syms = image_of(arr)
        if syms.max() >= (1 << 32):
            continue
        t = Text(arr)
        pats = [np.asarray(p, arr.dtype) for p in patterns(t, np.random.default_rng(len(name)))]
        top = 3 if name in K3_CASES else 2
        counts = [naive_counts(t, p, top) for p in pats]
        small = [q for q in range(len(pats)) if counts[q].sum() <= 20_000]   # located and compared occurrence by occurrence
        full = {q: naive(t, pats[q], top) for q in small}
        longest = int((t.ends - t.starts).max()) + 1
        rows = {}
        for flags in (AUTO, WALK, JUMP):
            with G.GrlGpu(0, flags) as ctx:
                ctx.fm_load(raw)
                for kmax in range(top + 1):
                    want = {q: [o for o in occ if o[2] <= kmax] for q, occ in full.items()}
                    if flags == AUTO:
                        hit_off, sp, ep, mm, info = ctx.fm_approx_count(pats, kmax)
                        check_hits(hit_off, sp, ep, mm, counts, kmax)
                        assert info["n_occ"] == sum(int(c[:kmax + 1].sum()) for c in counts) and (info["n_lf"] > 0 or not pats or t.ends.size == arr.size), (name, kmax)
                        if kmax == 0:   # the exact search, without its empty intervals
                            s0, e0, _ = ctx.fm_count(pats)
                            for q in range(len(pats)):
                                a, b = int(hit_off[q]), int(hit_off[q + 1])
                                assert list(zip(sp[a:b], ep[a:b])) == ([(s0[q], e0[q])] if e0[q] > s0[q] else []), (name, q)
                    sel = [q for q in small if flags != WALK or len(want[q]) * longest <= 20_000_000]
                    occ_off, ids, pos, mm, li = ctx.fm_approx_locate([pats[q] for q in sel], kmax)
                    assert li["n_occ"] == sum(len(want[q]) for q in sel) and li["n_hits"] >= 0
                    assert flags == AUTO or li["path"] == (0 if flags == WALK else 1) or li["n_occ"] == 0, (name, flags, li)
                    for i, q in enumerate(sel):
                        a, b = int(occ_off[i]), int(occ_off[i + 1])
                        got = list(zip(ids[a:b].tolist(), pos[a:b].tolist(), mm[a:b].tolist()))
                        assert sorted(got) == want[q], (name, flags, kmax, pats[q])
                        rows.setdefault((q, kmax), []).append(got)
        for key, lists in rows.items():
            assert all(x == lists[0] for x in lists), (name, key)


def test_k0_equals_exact(all_cases):
    arr = all_cases["reads_2000x150"]
    raw, _ = image_of(arr)
    t = Text(arr)
    pats = [np.asarray(p, np.uint8) for p in t.patterns(np.random.default_rng(4), n_hits=300, n_rand=100)]
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(raw)
        occ_off, ids, pos, _ = ctx.fm_locate(pats)
        a_off, a_ids, a_pos, a_mm, _ = ctx.fm_approx_locate(pats, 0)
        assert np.array_equal(occ_off, a_off) and np.array_equal(ids, a_ids) and np.array_equal(pos, a_pos) and not a_mm.any()


def test_exact_launches_unchanged(all_cases):
    """fm_count and fm_locate issue the launches they issued before the locate half became shared with the approximate search"""
    arr = all_cases["dna_500"]
    raw, _ = image_of(arr)
    pats = [np.frombuffer(b"ACG", np.uint8), np.frombuffer(b"TTA", np.uint8)]
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(raw)
        ctx.profile_enable(True)
        ctx.profile_reset()
        ctx.fm_count(pats)
        assert {k: v[0] for k, v in ctx.profile().items()} == {"fm_count": 1}
        ctx.profile_reset()
        ctx.fm_locate(pats)
        assert {k: v[0] for k, v in ctx.profile().items()} == {"fm_count": 2, "fm_occ_count": 1, "scan_single_block": 1, "fm_locate_walk": 1}


def test_batch_equals_chunks(all_cases):
    arr = all_cases["reads_2000x150"]
    raw, _ = image_of(arr)
    t = Text(arr)
    pats = [np.asarray(p, np.uint8) for p in patterns(t, np.random.default_rng(3), n_win=400, n_rand=100, max_len=20)]
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(raw)
        hit_off, sp, ep, mm, _ = ctx.fm_approx_count(pats, 2)
        occ_off, ids, pos, omm, _ = ctx.fm_approx_locate(pats, 2)
        for a in range(0, len(pats), 77):
            h2, s2, e2, m2, _ = ctx.fm_approx_count(pats[a:a + 77], 2)
            lo, hi = int(hit_off[a]), int(hit_off[min(a + 77, len(pats))])
            assert np.array_equal(s2, sp[lo:hi]) and np.array_equal(e2, ep[lo:hi]) and np.array_equal(m2, mm[lo:hi])
            assert np.array_equal(h2, hit_off[a:a + 78] - hit_off[a])
            o2, i2, p2, d2, _ = ctx.fm_approx_locate(pats[a:a + 77], 2)
            lo, hi = int(occ_off[a]), int(occ_off[min(a + 77, len(pats))])
            assert np.array_equal(i2, ids[lo:hi]) and np.array_equal(p2, pos[lo:hi]) and np.array_equal(d2, omm[lo:hi])


def test_pool_rerun(all_cases):
    """more hits than the first pool of the search (max(2^16, 4 n_pat)) and than the binding's first capacity: both calls rerun"""
    arr = all_cases["reads_100k"]
    raw, _ = image_of(arr)
    t = Text(arr)
    rng = np.random.default_rng(8)
    pats = [rng.choice(np.frombuffer(b"ACGT", np.uint8), 6) for _ in range(200)]
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(raw)
        hit_off, sp, ep, mm, info = ctx.fm_approx_count(pats, 3)
        assert info["n_hits"] > (1 << 16), info
        for q in rng.choice(len(pats), 3, replace=False):
            want = naive_counts(t, pats[q], 3)
            a, b = int(hit_off[q]), int(hit_off[q + 1])
            for x in range(4):
                assert int((ep[a:b] - sp[a:b])[mm[a:b] == x].sum()) == int(want[x]), (q, x)


@pytest.mark.parametrize("name,path", [("reads_1M", 0), ("rep_20x2M", 1)])
def test_at_scale(name, path):
    """build_bwt_packed of a 40-150 MB collection, 10^4 windows of 32 with 0 to 2 substitutions; counts against the pigeonhole
    oracle on a subset, locate on another"""
    import gen
    arr = {"reads_1M": lambda: gen.dna_reads(1_000_000, 150, seed=42), "rep_20x2M": lambda: gen.repetitive_genomes(20, 2_000_000, seed=7)}[name]()
    img = np.empty(16 + arr.size * 16, np.uint8)
    nb, _, _, _, _ = G.build_bwt_packed(arr, img, n_threads=8)
    t = Text(arr)
    rng = np.random.default_rng(5)
    starts = rng.integers(0, arr.size - 32, 10_000)
    win = arr[(starts[:, None] + np.arange(32)).ravel()].reshape(-1, 32)
    win = win[(win != t.sep).all(axis=1)]
    cells = mutate(rng, win, np.frombuffer(b"ACGT", np.uint8), rng.integers(0, 3, win.shape[0]))
    off = np.arange(0, cells.size + 1, 32, dtype=np.uint64)
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(img[:nb])
        hit_off, sp, ep, mm, info = ctx.fm_approx_count((cells.ravel(), off), 2)
        assert (hit_off[1:] > hit_off[:-1]).all()   # every mutated window is within 2 of where it came from
        for q in rng.choice(cells.shape[0], 10, replace=False):
            a, b = int(hit_off[q]), int(hit_off[q + 1])
            assert int((ep[a:b] - sp[a:b]).sum()) == len(pigeonhole(t, cells[q], 2)), q
        sub = rng.choice(cells.shape[0], 10, replace=False)
        occ_off, ids, pos, omm, li = ctx.fm_approx_locate([cells[q] for q in sub], 2)
        assert li["path"] == path, li
        for i, q in enumerate(sub):
            a, b = int(occ_off[i]), int(occ_off[i + 1])
            assert sorted(zip(ids[a:b].tolist(), pos[a:b].tolist(), omm[a:b].tolist())) == pigeonhole(t, cells[q], 2), q


def image_of_runs(syms, lens, sb=4, fb=4):
    from oracle import oracle as O
    return O.rl_bwt_bytes(np.asarray(syms, np.uint64), np.asarray(lens, np.uint64), sb, fb)


def test_errors(all_cases):
    arr = all_cases["dna_500"]
    raw, _ = image_of(arr)
    L = lib_gpu()
    info = FmApprox()
    cells, off = np.frombuffer(b"ACGTAC", np.uint8).copy(), np.array([0, 2, 6], np.uint64)
    hoff, se, mm, ids = np.zeros(3, np.uint64), np.zeros(64, np.uint64), np.zeros(64, np.uint8), np.zeros(64, np.uint32)
    P = (cells.ctypes.data, off.ctypes.data, 2, 1)

    def count(k, o=off, cap=32, w=1):
        return L.grlgpu_fm_approx_count(h, cells.ctypes.data, o.ctypes.data, 2, w, k, hoff.ctypes.data, se.ctypes.data, mm.ctypes.data, cap, C.byref(info))

    def locate(k, o=off, cap=64):
        return L.grlgpu_fm_approx_locate(h, cells.ctypes.data, o.ctypes.data, 2, 1, k, hoff.ctypes.data, ids.ctypes.data, ids.ctypes.data, mm.ctypes.data, cap,
                                         C.byref(info))
    with G.GrlGpu(0) as ctx:
        h = ctx._h
        assert count(1) == ERR_STATE and locate(1) == ERR_STATE   # no index
        ctx.fm_load(raw)
        assert count(4) == ERR_ARG and locate(4) == ERR_ARG
        for w in (0, 3, 16):
            assert count(1, w=w) == ERR_ARG
        for bad_off in ([1, 2, 6], [0, 2, 2], [0, 3, 2]):
            o = np.array(bad_off, np.uint64)
            assert count(1, o) == ERR_ARG and locate(1, o) == ERR_ARG
        assert L.grlgpu_fm_approx_count(h, *P, 1, None, se.ctypes.data, mm.ctypes.data, 8, C.byref(info)) == ERR_ARG   # null offsets
        assert L.grlgpu_fm_approx_count(h, None, None, 0, 1, 1, None, None, None, 0, C.byref(info)) == 0   # no patterns
        with pytest.raises(G.GrlGpuError) as e:
            ctx.fm_approx_count([b"AC"], 4)
        assert e.value.status == ERR_ARG
        # capacities: the number needed comes back
        _, sp, ep, _, d = ctx.fm_approx_count((cells, off), 1)
        assert d["n_hits"] > 1 and d["n_occ"] > 1
        assert count(1, cap=d["n_hits"] - 1) == ERR_ARG and info.n_hits == d["n_hits"]
        assert count(1, cap=d["n_hits"]) == 0
        assert locate(1, cap=d["n_occ"] - 1) == ERR_ARG and info.n_occ == d["n_occ"]
        ctx.fm_drop()
        with pytest.raises(G.GrlGpuError) as e:
            ctx.fm_approx_locate((cells, off), 1)
        assert e.value.status == ERR_STATE
    # run lists that are not a BWT: locating the hits meets the LF cycle without separator on every path
    from oracle import oracle as O
    for Lb in (np.array([1, 3, 2]), np.array([1, 4, 2, 3]), np.array([1, 2, 1, 4, 3, 5])):
        s, ln = O.rle(Lb)
        for flags in (WALK, JUMP, AUTO):
            with G.GrlGpu(0, flags) as ctx:
                ctx.fm_load(image_of_runs(s, ln))
                with pytest.raises(G.GrlGpuError) as e:
                    ctx.fm_approx_locate([np.array([c], np.uint8) for c in np.unique(Lb)[1:]], 1)
                assert e.value.status == ERR_ILL_FORMED, (Lb, flags)


@pytest.mark.parametrize("name", ["with_empty", "dna_500", "u16_small_sigma", "homopolymers_multi", "reads_2000x150"])
def test_tool_matches_fm_query(all_cases, tmp_path, name):
    arr = all_cases[name]
    raw, _ = image_of(arr)
    rl, pp = tmp_path / "x.rl_bwt", tmp_path / "p.bin"
    rl.write_bytes(raw)
    t = Text(arr)
    pats = [p for p in patterns(t, np.random.default_rng(11)) if t.sep not in p]
    w = arr.dtype.itemsize
    patterns_file(pp, pats, t.sep, w)
    for kmax in (0, 1, 2, 3):
        for loc in ([], ["-l"]):
            cmd = [str(rl), str(pp), "-a", str(w), "-k", str(kmax)] + loc
            host = subprocess.run([lib("fm_query")] + cmd, capture_output=True)
            dev = subprocess.run([lib("fm_query_gpu")] + cmd, capture_output=True)
            assert host.returncode == dev.returncode == 0 and dev.stdout == host.stdout, (name, kmax, loc, dev.stderr)
            assert len(host.stdout.splitlines()) == len(pats)
