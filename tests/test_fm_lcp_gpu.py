"""GPU suite: the LCP array on the device (grlgpu_fm_lcp, GrlGpu.fm_lcp, fm_lcp_gpu) against the host tool fm_lcp and the oracle
of lcp_oracle.py, on both paths, at scale, with the locate table shared with locate and extract, and its errors."""
import ctypes as C
import functools
import subprocess

import numpy as np
import pytest

import gen
import grlbwt_b200 as G
from extract_oracle import as_arrays, requests
from fm_oracle import Text, image_of, lib
from grlbwt_b200.api import FmLcp, lib_gpu
from lcp_oracle import Rows, lcp_of

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_ILL_FORMED, ERR_STATE, ERR_LIMIT = -1, -2, -5, -6
AUTO, WALK, JUMP = 0, G.FLAG_FORCE_WALK, G.FLAG_FORCE_JUMP


def host_lcp(img, tmp_path):
    rl, out = tmp_path / "x.rl_bwt", tmp_path / "host.bin"
    np.frombuffer(bytes(img), np.uint8).tofile(rl)
    r = subprocess.run([lib("fm_lcp"), str(rl), str(out)], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    return np.fromfile(out, "<u4")


def image_of_runs(syms, lens, sb=4, fb=4):
    from oracle import oracle as O
    return O.rl_bwt_bytes(np.asarray(syms, np.uint64), np.asarray(lens, np.uint64), sb, fb)


def test_every_case(all_cases, tmp_path):
    """every golden case: the device array equals fm_lcp's bytes on the automatic path and under FORCE_JUMP and FORCE_WALK;
    n_irreducible is the count of irreducible rows from the runs, sum_irreducible the oracle's LCP summed over them"""
    for name, arr in all_cases.items():
        raw, syms = image_of(arr)
        if syms.max() >= (1 << 32):   # beyond the device's 32-bit symbols
            with G.GrlGpu(0) as ctx, pytest.raises(G.GrlGpuError) as e:
                ctx.fm_load(raw)
            assert e.value.status == ERR_LIMIT, name
            continue
        want = host_lcp(raw, tmp_path)
        oracle, rows, _ = lcp_of(arr, raw, only=Rows.irreducible)
        irr = rows.irreducible()
        for flags in (AUTO, WALK, JUMP):
            with G.GrlGpu(0, flags) as ctx:
                ctx.fm_load(raw)
                got, info = ctx.fm_lcp()
            assert got.dtype == np.uint32 and np.array_equal(got, want), (name, flags)
            assert info["n"] == rows.n and info["n_irreducible"] == int(irr.sum()), (name, flags, info)
            assert info["sum_irreducible"] == int(oracle[irr].sum()), (name, flags, info)
            assert flags == AUTO or info["path"] == (0 if flags == WALK else 1), (name, flags, info)
            assert info["path"] == 1 or info["jump_rounds"] == 0


@functools.lru_cache(maxsize=None)
def scale_case(name):
    arr = {"reads_1M": lambda: gen.dna_reads(1_000_000, 150, seed=42), "rep_20x2M": lambda: gen.repetitive_genomes(20, 2_000_000, seed=7)}[name]()
    img = np.empty(16 + arr.size * 16, np.uint8)
    nb, _, _, _, _ = G.build_bwt_packed(arr, img, n_threads=8)
    return arr, img[:nb].copy()


@pytest.mark.parametrize("name,path", [("reads_1M", 0), ("rep_20x2M", 1)])
def test_at_scale(name, path, tmp_path):
    """150 MB of reads take the walk; 40 MB of genomes take the table, with long comparisons and the max carried across many
    scan tiles; both equal the host tool"""
    arr, img = scale_case(name)
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(img)
        got, info = ctx.fm_lcp()
        assert info["path"] == path and (info["jump_rounds"] > 0) == (path == 1), info
        again, info2 = ctx.fm_lcp()   # a second call: the same array, and the table once built is not built again
        assert info2["path"] == path and info2["jump_rounds"] == 0 and np.array_equal(again, got)
    want = host_lcp(img, tmp_path)
    assert np.array_equal(got, want), name
    assert info["n"] == arr.size and info["n_irreducible"] < arr.size


def test_shared_table():
    """after a locate that built the locate table, LCP uses it without building it again; after an LCP call that built it,
    extract does not build it either"""
    arr, img = scale_case("rep_20x2M")
    t = Text(arr)
    pats = [arr[t.starts[3] + 1000: t.starts[3] + 1032], arr[t.starts[7] + 5: t.starts[7] + 25]]
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(img)
        *_, li = ctx.fm_locate(pats)
        assert li["path"] == 1 and li["jump_rounds"] > 0, li
        first, info = ctx.fm_lcp()
        assert info["path"] == 1 and info["jump_rounds"] == 0, info
        ctx.fm_load(img)   # drops the table
        second, info = ctx.fm_lcp()
        assert info["path"] == 1 and info["jump_rounds"] > 0, info
        assert np.array_equal(first, second)
        *_, xi = ctx.fm_extract([0, 5], [10, 20], [30, 40])
        assert xi["path"] == 1 and xi["jump_rounds"] == 0, xi


def test_queries_unchanged(all_cases):
    """count, locate and extract answer the same before and after an LCP call, and a load launches what it launched before"""
    arr = all_cases["reads_2000x150"]
    raw, _ = image_of(arr)
    t = Text(arr)
    pats = [np.asarray(p, np.uint8) for p in t.patterns(np.random.default_rng(5), n_hits=60, n_rand=20)]
    reqs = as_arrays(requests(t, np.random.default_rng(6)))

    def answers(ctx):
        sp, ep, _ = ctx.fm_count(pats)
        occ_off, ids, pos, _ = ctx.fm_locate(pats)
        off, cells, _ = ctx.fm_extract(*reqs)
        return [x.tobytes() for x in (sp, ep, occ_off, ids, pos, off, cells)]

    with G.GrlGpu(0) as ctx:
        ctx.profile_enable(True)
        ctx.profile_reset()
        ctx.fm_load(raw)
        load = {k: v[0] for k, v in ctx.profile().items()}
        before = answers(ctx)
        ctx.fm_lcp()
        assert answers(ctx) == before
        ctx.profile_reset()
        ctx.fm_load(raw)
        assert {k: v[0] for k, v in ctx.profile().items()} == load
        assert not any(k.startswith("fm_lcp") for k in load)
        ctx.fm_lcp()
        assert answers(ctx) == before


def test_errors(all_cases):
    arr = all_cases["dna_500"]
    raw, _ = image_of(arr)
    n = arr.size
    L = lib_gpu()
    info = FmLcp()
    out = np.full(n, 0xABABABAB, np.uint32)

    def call(h, dst=out, cap=n):
        return L.grlgpu_fm_lcp(h, None if dst is None else dst.ctypes.data, cap, C.byref(info))
    with G.GrlGpu(0) as ctx:
        h = ctx._h
        assert call(h) == ERR_STATE   # no index yet
        ctx.fm_load(raw)
        assert call(h, dst=None, cap=0) == ERR_ARG and info.n == n
        assert call(h, dst=None, cap=n) == ERR_ARG and info.n == n
        assert call(h, cap=n - 1) == ERR_ARG and info.n == n and (out == 0xABABABAB).all()
        assert call(h) == 0 and info.n == n and out[0] == 0
        ctx.fm_drop()
        assert call(h) == ERR_STATE
        with pytest.raises(G.GrlGpuError) as e:
            ctx.fm_lcp()
        assert e.value.status == ERR_STATE
    # run lists that are not a BWT (LF has a cycle without separator): both paths refuse them
    for Lb in (np.array([1, 3, 2]), np.array([1, 4, 2, 3]), np.array([1, 2, 1, 4, 3, 5])):
        from oracle import oracle as O
        s, lens = O.rle(Lb)
        img = image_of_runs(s, lens)
        for flags in (AUTO, WALK, JUMP):
            with G.GrlGpu(0, flags) as ctx:
                ctx.fm_load(img)
                with pytest.raises(G.GrlGpuError) as e:
                    ctx.fm_lcp()
                assert e.value.status == ERR_ILL_FORMED, (Lb, flags)


@pytest.mark.parametrize("name", ["with_empty", "dna_500", "u16_small_sigma", "homopolymers_multi", "reads_2000x150"])
def test_tool_matches_fm_lcp(all_cases, tmp_path, name):
    raw, _ = image_of(all_cases[name])
    rl, ho, do = tmp_path / "x.rl_bwt", tmp_path / "host.bin", tmp_path / "dev.bin"
    rl.write_bytes(raw)
    for tool, dst in (("fm_lcp", ho), ("fm_lcp_gpu", do)):
        r = subprocess.run([lib(tool), str(rl), str(dst)], capture_output=True)
        assert r.returncode == 0, (tool, r.stderr.decode())
    assert do.read_bytes() == ho.read_bytes() and len(ho.read_bytes()) == 4 * all_cases[name].size, name
