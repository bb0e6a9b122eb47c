"""GPU suite: extract on the device (grlgpu_fm_extract, GrlGpu.fm_extract, fm_extract_gpu) against numpy slices of the collections,
the device inversion, locate, and the host tool fm_extract."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import gen
import grlbwt_b200 as G
from extract_oracle import U32_MAX, as_arrays, expected, requests, requests_file, tool_output
from fm_oracle import Text, image_of, lib
from grlbwt_b200.api import FmExtract, lib_gpu

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_ILL_FORMED, ERR_STATE, ERR_LIMIT = -1, -2, -5, -6
AUTO, WALK, JUMP = 0, G.FLAG_FORCE_WALK, G.FLAG_FORCE_JUMP


def pieces(out_off, cells):
    return [cells[int(out_off[q]):int(out_off[q + 1])] for q in range(out_off.size - 1)]


def image_of_runs(syms, lens, sb=4, fb=4):
    from oracle import oracle as O
    return O.rl_bwt_bytes(np.asarray(syms, np.uint64), np.asarray(lens, np.uint64), sb, fb)


def test_every_case(all_cases):
    """every golden case: the request set of the CPU test on the three paths, which agree byte for byte"""
    for name, arr in all_cases.items():
        raw, syms = image_of(arr)
        if syms.max() >= (1 << 32):   # beyond the device's 32-bit symbols
            with G.GrlGpu(0) as ctx, pytest.raises(G.GrlGpuError) as e:
                ctx.fm_load(raw)
            assert e.value.status == ERR_LIMIT, name
            continue
        t, w = Text(arr), arr.dtype.itemsize
        reqs = requests(t, np.random.default_rng(len(name)))
        want = expected(t, reqs)
        got = []
        for flags in (AUTO, WALK, JUMP):
            with G.GrlGpu(0, flags) as ctx:
                ctx.fm_load(raw)
                off, cells, info = ctx.fm_extract(*as_arrays(reqs), cell_bytes=w)
            assert info["n_req"] == len(reqs) and info["n_cells"] == sum(x.size for x in want), (name, info)
            assert flags == AUTO or info["path"] == (0 if flags == WALK else 1), (name, flags, info)
            assert cells.dtype == arr.dtype
            for q, x in enumerate(pieces(off, cells)):
                assert np.array_equal(x, want[q]), (name, flags, reqs[q])
            got.append((off.tobytes(), cells.tobytes()))
        assert got[0] == got[1] == got[2], name


def test_whole_strings_equal_invert(all_cases):
    """(k, 0, to the end) for every k, at every cell width, is ctx.invert(raw, w) without the separators"""
    for name, arr in all_cases.items():
        raw, syms = image_of(arr)
        if syms.max() >= (1 << 32):
            continue
        t = Text(arr)
        keep = np.ones(arr.size, bool)
        keep[t.ends] = False
        ids = np.arange(t.ends.size)
        with G.GrlGpu(0) as ctx:
            ctx.fm_load(raw)
            for w in (1, 2, 4, 8):
                inv, _ = ctx.invert(raw, w)
                off, cells, _ = ctx.fm_extract(ids, 0, None, w)
                assert np.array_equal(cells, inv[keep]), (name, w)
                assert np.array_equal(np.diff(off.astype(np.int64)), t.ends - t.starts), (name, w)


@pytest.mark.parametrize("name", ["dna_500", "reads_2000x150", "u16_small_sigma", "rep_50x200k"])
def test_locate_then_extract(all_cases, name):
    """each occurrence (k, p) of P that fm_locate returns extracts back to P, its arrays passed straight in; windows around it
    match the collection"""
    arr = all_cases[name]
    raw, _ = image_of(arr)
    t = Text(arr)
    pats = [np.asarray(p, arr.dtype) for p in t.patterns(np.random.default_rng(2), n_hits=60, n_rand=20)]
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(raw)
        occ_off, ids, pos, _ = ctx.fm_locate(pats)
        m = np.repeat([p.size for p in pats], np.diff(occ_off.astype(np.int64)))
        assert ids.dtype == pos.dtype == np.uint32 and ids.size > 0
        off, cells, _ = ctx.fm_extract(ids, pos, m.astype(np.uint32), arr.dtype.itemsize)
        got = pieces(off, cells)
        for q in range(len(pats)):
            for o in range(int(occ_off[q]), int(occ_off[q + 1])):
                assert np.array_equal(got[o], pats[q]), (name, q, o)
        lo = np.maximum(pos.astype(np.int64) - 10, 0)
        off, cells, _ = ctx.fm_extract(ids, lo, m + 20, arr.dtype.itemsize)
        want = expected(t, list(zip(ids.tolist(), lo.tolist(), (m + 20).tolist())))
        for o, x in enumerate(pieces(off, cells)):
            assert np.array_equal(x, want[o]), (name, o)


def random_requests(t, rng, n):
    lens = t.ends - t.starts
    k = rng.integers(0, lens.size, n)
    f = (rng.random(n) * (lens[k] + 2)).astype(np.int64)
    m = rng.integers(0, 400, n)
    m[rng.random(n) < 0.1] = U32_MAX
    return k, f, m


def check_against_numpy(t, k, f, m, off, cells):
    lo = t.starts[k] + np.minimum(f, t.ends[k] - t.starts[k])
    hi = np.minimum(t.starts[k] + f + np.minimum(m, 1 << 40), t.ends[k])
    cnt = np.maximum(hi - lo, 0)
    assert np.array_equal(np.diff(off.astype(np.int64)), cnt)
    idx = np.repeat(lo - np.concatenate(([0], np.cumsum(cnt)[:-1])), cnt) + np.arange(int(cnt.sum()))
    assert np.array_equal(cells, t.arr[idx])


def scale_case(name):
    arr = {"reads_1M": lambda: gen.dna_reads(1_000_000, 150, seed=42), "rep_20x2M": lambda: gen.repetitive_genomes(20, 2_000_000, seed=7)}[name]()
    img = np.empty(16 + arr.size * 16, np.uint8)
    nb, _, _, _, _ = G.build_bwt_packed(arr, img, n_threads=8)
    return arr, img[:nb]


@pytest.mark.parametrize("name,path", [("reads_1M", 0), ("rep_20x2M", 1)])
def test_at_scale(name, path):
    """build_bwt_packed of a 40-150 MB collection, 10^5 random requests against numpy; reads take the walk, genomes the samples"""
    arr, img = scale_case(name)
    t = Text(arr)
    k, f, m = random_requests(t, np.random.default_rng(9), 100_000)
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(img)
        off, cells, info = ctx.fm_extract(k, f, m)
        assert info["path"] == path, info
        check_against_numpy(t, k, f, m, off, cells)
        off2, cells2, info2 = ctx.fm_extract(k, f, m)   # a second call: the same answer (from the samples once built)
        assert info2["path"] == path and info2["jump_rounds"] == 0
        assert np.array_equal(off2, off) and np.array_equal(cells2, cells)


def test_shared_table():
    """locate and extract build the locate table once between them; a fresh load drops it and the samples"""
    arr, img = scale_case("rep_20x2M")
    t = Text(arr)
    pats = [arr[t.starts[3] + 1000: t.starts[3] + 1032], arr[t.starts[7] + 5: t.starts[7] + 25]]
    k, f, m = random_requests(t, np.random.default_rng(4), 1000)
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(img)
        *_, li = ctx.fm_locate(pats)
        assert li["path"] == 1 and li["jump_rounds"] > 0, li
        off, cells, xi = ctx.fm_extract(k, f, m)
        assert xi["path"] == 1 and xi["jump_rounds"] == 0, xi
        check_against_numpy(t, k, f, m, off, cells)
        ctx.fm_load(img)   # drops the table and the samples
        off, cells, xi = ctx.fm_extract(k, f, m)
        assert xi["path"] == 1 and xi["jump_rounds"] > 0, xi
        check_against_numpy(t, k, f, m, off, cells)
        *_, li = ctx.fm_locate(pats)
        assert li["path"] == 1 and li["jump_rounds"] == 0, li


def test_errors(all_cases, tmp_path):
    arr = all_cases["dna_500"]
    raw, _ = image_of(arr)
    N = Text(arr).ends.size
    L = lib_gpu()
    info = FmExtract()
    ids, frm, ln = np.array([0, 1], np.uint32), np.array([2, 0], np.uint32), np.array([5, U32_MAX], np.uint32)
    off, out = np.zeros(3, np.uint64), np.zeros(4096, np.uint8)
    p = lambda a: a.ctypes.data   # noqa: E731

    def call(h, i=ids, f=frm, n=ln, n_req=2, w=1, o=off, dst=out, cap=4096):
        return L.grlgpu_fm_extract(h, None if i is None else p(i), None if f is None else p(f), None if n is None else p(n), n_req, w,
                                   None if o is None else p(o), None if dst is None else p(dst), cap, C.byref(info))
    with G.GrlGpu(0) as ctx:
        h = ctx._h
        assert call(h) == ERR_STATE   # no index yet
        ctx.fm_load(raw)
        for w in (0, 3, 16):
            assert call(h, w=w) == ERR_ARG
        for kw in (dict(i=None), dict(f=None), dict(n=None), dict(o=None), dict(dst=None)):
            assert call(h, **kw) == ERR_ARG, kw
        assert call(h, i=np.array([0, N], np.uint32)) == ERR_ARG   # k = N
        assert call(h, n_req=1 << 32) == ERR_LIMIT   # 2^32 requests: refused before any array is read
        assert call(h, i=None, f=None, n=None, n_req=0, o=None, dst=None, cap=0) == 0   # no requests
        assert call(h, cap=0, dst=None) == ERR_ARG and info.n_cells > 1   # capacity: the number needed comes back
        need = info.n_cells
        out[:] = 0xAB
        assert call(h, cap=need - 1) == ERR_ARG and info.n_cells == need and (out == 0xAB).all()
        assert call(h, cap=need) == 0 and info.n_cells == need
        ctx.fm_drop()
        assert call(h) == ERR_STATE
        with pytest.raises(G.GrlGpuError) as e:
            ctx.fm_extract([0])
        assert e.value.status == ERR_STATE
    # run lists that are not a BWT (LF has a cycle without separator): the samples need the locate table and fail; a walk from
    # row k always ends and writes what the host tool writes
    for Lb in (np.array([1, 3, 2]), np.array([1, 4, 2, 3]), np.array([1, 2, 1, 4, 3, 5])):
        from oracle import oracle as O
        s, lens = O.rle(Lb)
        img = image_of_runs(s, lens)
        n_str = int((Lb == 1).sum())
        reqs = [(k, None, None) for k in range(n_str)] + [(k, 1, 2) for k in range(n_str)]
        with G.GrlGpu(0, JUMP) as ctx:
            ctx.fm_load(img)
            with pytest.raises(G.GrlGpuError) as e:
                ctx.fm_extract(*as_arrays(reqs))
            assert e.value.status == ERR_ILL_FORMED, Lb
        with G.GrlGpu(0, WALK) as ctx:
            ctx.fm_load(img)
            off, cells, info = ctx.fm_extract(*as_arrays(reqs))
            assert info["path"] == 0
        rl, rq, ho = tmp_path / "x.rl_bwt", tmp_path / "req.txt", tmp_path / "host.bin"
        rl.write_bytes(img)
        requests_file(rq, reqs)
        r = subprocess.run([lib("fm_extract"), str(rl), str(rq), str(ho)], capture_output=True)
        assert r.returncode == 0, r.stderr
        dev = b"".join(x.tobytes() + b"\x01" for x in pieces(off, cells))
        assert dev == ho.read_bytes(), Lb


def test_context_is_left_untouched(all_cases):
    """extract calls between rounds change neither the rounds nor a later inversion"""
    a, b = all_cases["mutated_200x5k"], all_cases["reads_2000x150"]
    raw, _ = image_of(a)
    t = Text(a)
    reqs = as_arrays(requests(t, np.random.default_rng(1)))
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
        first = ctx.fm_extract(*reqs)
        ctx.set_text(b)
        got = []
        while True:
            r = ctx.round()
            again = ctx.fm_extract(*reqs)
            assert np.array_equal(again[0], first[0]) and np.array_equal(again[1], first[1])
            got.append((ctx.fetch_parse().copy(), ctx.level_checksum()))
            if r.done:
                break
        inv, _ = ctx.invert(raw)
        assert inv.tobytes() == a.tobytes()
    assert len(got) == len(want)
    for (p1, c1), (p2, c2) in zip(got, want):
        assert np.array_equal(p1, p2) and c1 == c2


@pytest.mark.parametrize("name", ["with_empty", "dna_500", "u16_small_sigma", "homopolymers_multi", "reads_2000x150"])
def test_tool_matches_fm_extract(all_cases, tmp_path, name):
    arr = all_cases[name]
    raw, _ = image_of(arr)
    t, w = Text(arr), arr.dtype.itemsize
    rl, rq, ho, do = tmp_path / "x.rl_bwt", tmp_path / "req.txt", tmp_path / "host.bin", tmp_path / "dev.bin"
    rl.write_bytes(raw)
    reqs = requests(t, np.random.default_rng(11)) + [(0, 1 << 40, None), (0, 0, 1 << 40)]   # from and len beyond 32 bits
    requests_file(rq, reqs)
    for tool, dst in (("fm_extract", ho), ("fm_extract_gpu", do)):
        r = subprocess.run([lib(tool), str(rl), str(rq), str(dst), "-a", str(w)], capture_output=True)
        assert r.returncode == 0, (tool, r.stderr.decode())
    assert do.read_bytes() == ho.read_bytes() == tool_output(t, reqs, w), name
