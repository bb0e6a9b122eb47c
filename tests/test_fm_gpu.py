"""GPU suite: the FM-index on the device (grlgpu_fm_load / _count / _locate / _drop, GrlGpu.fm_*, fm_query_gpu) against a naive
find over the collections and the host tool fm_query."""
import ctypes as C

import numpy as np
import pytest

import grlbwt_b200 as G
from fm_oracle import Text, image_of, lib, patterns_file, run_tool
from grlbwt_b200.api import FmQuery, lib_gpu

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_ILL_FORMED, ERR_STATE, ERR_LIMIT = -1, -2, -5, -6
AUTO, WALK, JUMP = 0, G.FLAG_FORCE_WALK, G.FLAG_FORCE_JUMP


def as_pairs(occ_off, ids, pos, q):
    a, b = int(occ_off[q]), int(occ_off[q + 1])
    return list(zip(ids[a:b].tolist(), pos[a:b].tolist()))


def case_patterns(t, arr, seed):
    pats = t.patterns(np.random.default_rng(seed))
    alpha = np.unique(arr[arr != t.sep])
    pats.append([t.sep])                                   # the separator alone and inside patterns: no occurrence
    if alpha.size:
        pats += [[int(alpha[0]), t.sep], [t.sep, int(alpha[-1])]]
    return [np.asarray(p, arr.dtype) for p in pats]


def test_every_case(all_cases):
    """every golden case: counts and sorted locate lists of the oracle on the three locate paths, which agree row for row"""
    for name, arr in all_cases.items():
        raw, syms = image_of(arr)
        if syms.max() >= (1 << 32):   # beyond the device's 32-bit symbols
            with G.GrlGpu(0) as ctx, pytest.raises(G.GrlGpuError) as e:
                ctx.fm_load(raw)
            assert e.value.status == ERR_LIMIT, name
            continue
        t = Text(arr)
        pats = case_patterns(t, arr, len(name))
        want = [t.occurrences(p) for p in pats]
        longest = int((t.ends - t.starts).max()) + 1
        rows = {}
        for flags in (AUTO, WALK, JUMP):
            with G.GrlGpu(0, flags) as ctx:
                info = ctx.fm_load(raw)
                assert info["n"] == arr.size and info["n_strings"] == t.ends.size and info["sep"] == t.sep, (name, info)
                sp, ep, _ = ctx.fm_count(pats)
                assert (ep - sp).tolist() == [len(w) for w in want], (name, flags)
                assert all(sp[q] == ep[q] == 0 for q in range(len(pats)) if not want[q]), name
                # the forced walk follows every occurrence through its whole string: only the patterns where that stays small
                sel = [q for q in range(len(pats)) if flags != WALK or len(want[q]) * longest <= 20_000_000]
                occ_off, ids, pos, li = ctx.fm_locate([pats[q] for q in sel])
                assert li["n_occ"] == sum(len(want[q]) for q in sel)
                assert flags == AUTO or li["path"] == (0 if flags == WALK else 1) or li["n_occ"] == 0, (name, flags, li)
                for i, q in enumerate(sel):
                    got = as_pairs(occ_off, ids, pos, i)
                    assert sorted(got) == want[q], (name, flags, pats[q])
                    rows.setdefault(q, []).append(got)
        for q, lists in rows.items():   # row order: the paths agree entry for entry
            assert all(x == lists[0] for x in lists), (name, pats[q])


def test_batch_equals_chunks(all_cases):
    arr = all_cases["reads_2000x150"]
    raw, _ = image_of(arr)
    t = Text(arr)
    pats = [np.asarray(p, np.uint8) for p in t.patterns(np.random.default_rng(3), n_hits=500, n_rand=500)]
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(raw)
        sp, ep, _ = ctx.fm_count(pats)
        for a in range(0, len(pats), 77):
            s2, e2, _ = ctx.fm_count(pats[a:a + 77])
            assert np.array_equal(s2, sp[a:a + 77]) and np.array_equal(e2, ep[a:a + 77])
        occ_off, ids, pos, _ = ctx.fm_locate(pats)
        for a in range(0, len(pats), 101):
            o2, i2, p2, _ = ctx.fm_locate(pats[a:a + 101])
            lo, hi = int(occ_off[a]), int(occ_off[min(a + 101, len(pats))])
            assert np.array_equal(i2, ids[lo:hi]) and np.array_equal(p2, pos[lo:hi]) and np.array_equal(o2, occ_off[a:a + 102] - occ_off[a])


@pytest.mark.parametrize("name,path", [("reads_1M", 0), ("rep_20x2M", 1)])
def test_at_scale(name, path):
    """build_bwt_packed of a 40-150 MB collection, 10^5 patterns; counts against the oracle on a subset, locate on another"""
    import gen
    arr = {"reads_1M": lambda: gen.dna_reads(1_000_000, 150, seed=42), "rep_20x2M": lambda: gen.repetitive_genomes(20, 2_000_000, seed=7)}[name]()
    img = np.empty(16 + arr.size * 16, np.uint8)
    nb, _, _, _, _ = G.build_bwt_packed(arr, img, n_threads=8)
    t = Text(arr)
    rng = np.random.default_rng(5)
    starts = rng.integers(0, arr.size - 32, 100_000)
    cells = arr[(starts[:, None] + np.arange(32)).ravel()].reshape(-1, 32)
    hit = (cells != t.sep).all(axis=1)
    cells[~hit] = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=(int((~hit).sum()), 32))
    off = np.arange(0, cells.size + 1, 32, dtype=np.uint64)
    with G.GrlGpu(0) as ctx:
        info = ctx.fm_load(img[:nb])
        assert info["n"] == arr.size
        sp, ep, _ = ctx.fm_count((cells.ravel(), off))
        assert (ep[hit] > sp[hit]).all()
        for q in rng.choice(cells.shape[0], 60, replace=False):
            assert ep[q] - sp[q] == len(t.occurrences(cells[q])), q
        sub = rng.choice(cells.shape[0], 20, replace=False)
        occ_off, ids, pos, li = ctx.fm_locate([cells[q] for q in sub])
        assert li["path"] == path, li
        for i, q in enumerate(sub):
            assert sorted(as_pairs(occ_off, ids, pos, i)) == t.occurrences(cells[q]), q


def test_errors(all_cases):
    arr = all_cases["dna_500"]
    raw, _ = image_of(arr)
    L = lib_gpu()
    info = FmQuery()
    cells, off = np.frombuffer(b"ACGTAC", np.uint8).copy(), np.array([0, 2, 6], np.uint64)
    buf, ids = np.zeros(8, np.uint64), np.zeros(64, np.uint32)
    with G.GrlGpu(0) as ctx:
        h = ctx._h
        # no index yet, and after a drop
        assert L.grlgpu_fm_count(h, cells.ctypes.data, off.ctypes.data, 2, 1, buf.ctypes.data, C.byref(info)) == ERR_STATE
        assert L.grlgpu_fm_locate(h, cells.ctypes.data, off.ctypes.data, 2, 1, buf.ctypes.data, ids.ctypes.data, ids.ctypes.data, 64, C.byref(info)) == ERR_STATE
        for bad in (raw[:-1], raw[:16], (0).to_bytes(8, "little") + raw[8:]):
            with pytest.raises(G.GrlGpuError) as e:
                ctx.fm_load(bad)
            assert e.value.status == ERR_ARG
        ctx.fm_load(raw)
        for w in (0, 3, 16):
            assert L.grlgpu_fm_count(h, cells.ctypes.data, off.ctypes.data, 2, w, buf.ctypes.data, C.byref(info)) == ERR_ARG
        for bad_off in ([1, 2, 6], [0, 2, 2], [0, 3, 2]):
            o = np.array(bad_off, np.uint64)
            assert L.grlgpu_fm_count(h, cells.ctypes.data, o.ctypes.data, 2, 1, buf.ctypes.data, C.byref(info)) == ERR_ARG
            assert L.grlgpu_fm_locate(h, cells.ctypes.data, o.ctypes.data, 2, 1, buf.ctypes.data, ids.ctypes.data, ids.ctypes.data, 64, C.byref(info)) == ERR_ARG
        assert L.grlgpu_fm_count(h, None, None, 0, 1, None, C.byref(info)) == 0   # no patterns
        # capacity: the number needed comes back
        sp, ep, _ = ctx.fm_count((cells, off))
        need = int((ep - sp).sum())
        assert need > 1
        rc = L.grlgpu_fm_locate(h, cells.ctypes.data, off.ctypes.data, 2, 1, buf.ctypes.data, ids.ctypes.data, ids.ctypes.data, need - 1, C.byref(info))
        assert rc == ERR_ARG and info.n_occ == need
        ctx.fm_drop()
        with pytest.raises(G.GrlGpuError) as e:
            ctx.fm_count((cells, off))
        assert e.value.status == ERR_STATE
        # a symbol of 2^32 or more
        with pytest.raises(G.GrlGpuError) as e:
            ctx.fm_load(image_of_runs([1, 1 << 32, 2], [1, 1, 1], 5, 1))
        assert e.value.status == ERR_LIMIT
    # run lists that are not a BWT: LF has a cycle without separator; locating every symbol meets it on every path
    for Lb in (np.array([1, 3, 2]), np.array([1, 4, 2, 3]), np.array([1, 2, 1, 4, 3, 5])):
        from oracle import oracle as O
        s, ln = O.rle(Lb)
        for flags in (WALK, JUMP, AUTO):
            with G.GrlGpu(0, flags) as ctx:
                ctx.fm_load(image_of_runs(s, ln))
                with pytest.raises(G.GrlGpuError) as e:
                    ctx.fm_locate([np.array([c], np.uint8) for c in np.unique(Lb)[1:]])
                assert e.value.status == ERR_ILL_FORMED, (Lb, flags)


def image_of_runs(syms, lens, sb=4, fb=4):
    from oracle import oracle as O
    return O.rl_bwt_bytes(np.asarray(syms, np.uint64), np.asarray(lens, np.uint64), sb, fb)


def test_context_is_left_untouched(all_cases):
    """an index on a context between rounds changes neither the rounds nor a later inversion; a second load replaces the first"""
    a, b, c = all_cases["mutated_200x5k"], all_cases["reads_2000x150"], all_cases["dna_500"]
    raw, _ = image_of(a)
    raw_c, _ = image_of(c)
    pats = [np.asarray(p, np.uint8) for p in Text(a).patterns(np.random.default_rng(1))]
    with G.GrlGpu(0) as ref:
        ref.set_text(b)
        want = []
        while True:
            r = ref.round()
            want.append((ref.fetch_parse().copy(), ref.level_checksum()))
            if r.done:
                break
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(raw)
        first = ctx.fm_locate(pats)
        ctx.set_text(b)
        got = []
        while True:
            r = ctx.round()
            again = ctx.fm_locate(pats)
            assert all(np.array_equal(x, y) for x, y in zip(again[:3], first[:3]))
            got.append((ctx.fetch_parse().copy(), ctx.level_checksum()))
            if r.done:
                break
        inv, _ = ctx.invert(raw)
        assert inv.tobytes() == a.tobytes()
        info = ctx.fm_load(raw_c)   # replaces the first index
        assert info["n"] == c.size
        sp, ep, _ = ctx.fm_count([np.frombuffer(b"ACG", np.uint8)])
        assert int(ep[0] - sp[0]) == len(Text(c).occurrences(np.frombuffer(b"ACG", np.uint8)))
        ctx.fm_drop()
        inv, _ = ctx.invert(raw)
        assert inv.tobytes() == a.tobytes()
    assert len(got) == len(want)
    for (p1, c1), (p2, c2) in zip(got, want):
        assert np.array_equal(p1, p2) and c1 == c2


@pytest.mark.parametrize("name", ["with_empty", "dna_500", "u16_small_sigma", "homopolymers_multi", "reads_2000x150"])
def test_tool_matches_fm_query(all_cases, tmp_path, name):
    arr = all_cases[name]
    raw, _ = image_of(arr)
    rl, pp = tmp_path / "x.rl_bwt", tmp_path / "p.bin"
    rl.write_bytes(raw)
    t = Text(arr)
    pats = t.patterns(np.random.default_rng(11), n_rand=10)
    w = arr.dtype.itemsize
    patterns_file(pp, pats, t.sep, w)
    for loc in (False, True):
        host = run_tool(lib("fm_query"), rl, pp, w, loc)
        assert run_tool(lib("fm_query_gpu"), rl, pp, w, loc) == host, (name, loc)
        assert len(host.splitlines()) == len(pats)
