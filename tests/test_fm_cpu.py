"""CPU suite: the host search tool fm_query against a naive find over the collections, both tools' usage, and the argument
checks of GrlGpu.fm_count / fm_locate (no device needed)."""
import subprocess

import numpy as np
import pytest

import gen
import grlbwt_b200 as G
from fm_oracle import Text, image_of, lib, parse_output, patterns_file, run_tool
from grlbwt_b200.api import _fm_patterns


def check_host_tool(arr, tmp_path, seed):
    """counts of every pattern; locate of the patterns whose walks stay small (each occurrence walks its whole string on the host)"""
    raw, _ = image_of(arr)
    rl, pp = tmp_path / "x.rl_bwt", tmp_path / "p.bin"
    rl.write_bytes(raw)
    t, w = Text(arr), arr.dtype.itemsize
    pats = t.patterns(np.random.default_rng(seed))
    want = [t.occurrences(p) for p in pats]
    patterns_file(pp, pats, t.sep, w)
    counts = parse_output(run_tool(lib("fm_query"), rl, pp, w, False))
    assert [c for c, _ in counts] == [len(x) for x in want] and not any(o for _, o in counts)
    longest = int((t.ends - t.starts).max()) + 1
    small = [q for q in range(len(pats)) if len(want[q]) * longest <= 2_000_000]
    patterns_file(pp, [pats[q] for q in small], t.sep, w)
    got = parse_output(run_tool(lib("fm_query"), rl, pp, w, True))
    assert len(got) == len(small)
    for q, (cnt, occ) in zip(small, got):
        assert cnt == len(want[q]) and sorted(occ) == want[q], pats[q]


@pytest.mark.parametrize("name", list(gen.small_cases()))
def test_fm_query_small_cases(name, tmp_path):
    check_host_tool(gen.small_cases()[name], tmp_path, 7)


def test_fm_query_fuzz(tmp_path):
    for i, (name, arr) in enumerate(gen.fuzz_cases()):
        check_host_tool(arr, tmp_path, i)


def test_fm_query_pattern_file_rules(tmp_path):
    arr = gen.small_cases()["with_empty"]
    raw, _ = image_of(arr)
    rl, pp = tmp_path / "x.rl_bwt", tmp_path / "p.bin"
    rl.write_bytes(raw)
    pp.write_bytes(b"AC\nT")   # the last pattern has no separator and still counts
    assert run_tool(lib("fm_query"), rl, pp, 1, False) == b"3\n6\n"
    for bad in (b"AC\n\nT\n", b"\nAC\n"):   # an empty pattern
        pp.write_bytes(bad)
        for tool in ("fm_query", "fm_query_gpu"):
            r = subprocess.run([lib(tool), str(rl), str(pp)], capture_output=True, text=True)
            if tool == "fm_query":
                assert r.returncode == 1 and "empty" in r.stderr
            else:   # without a device it fails earlier; either way with status 1
                assert r.returncode == 1


@pytest.mark.parametrize("tool", ["fm_query", "fm_query_gpu"])
def test_usage(tool):
    r = subprocess.run([lib(tool)], capture_output=True, text=True)
    assert r.returncode == 0 and "usage:" in r.stdout


@pytest.mark.parametrize("patterns", [
    [b"AC", b""],                                                  # an empty pattern
    [np.array([1, 2], np.uint8), np.array([1], np.uint16)],       # mixed cell types
    [np.zeros((2, 2), np.uint8)],                                  # not 1-d
    [np.array([1.0, 2.0])],                                        # not an unsigned cell type
    (np.array([1, 2, 3], np.uint8), np.array([1, 3])),             # offsets not from 0
    (np.array([1, 2, 3], np.uint8), np.array([0, 2, 2, 3])),       # an empty pattern
    (np.array([1, 2, 3], np.uint8), np.array([0, 4])),             # past the cells
    (np.array([1, 2, 3], np.uint8), np.array([0, -1, 3])),         # negative
    (np.array([1, 2, 3], np.uint8),),                              # not a pair
    "AC",                                                          # neither a list nor a pair
])
def test_pattern_argument_checks(patterns):
    with pytest.raises(G.GrlGpuError) as e:
        _fm_patterns(patterns)
    assert e.value.status == -1


def test_pattern_forms_agree():
    c1, o1 = _fm_patterns([b"AC", b"GTT", b"A"])
    c2, o2 = _fm_patterns((np.frombuffer(b"ACGTTA", np.uint8), np.array([0, 2, 5, 6])))
    assert c1.dtype == c2.dtype == np.uint8 and np.array_equal(c1, c2) and np.array_equal(o1, o2)
    c3, o3 = _fm_patterns([np.array([7, 8], np.uint32)])
    assert c3.dtype == np.uint32 and o3.tolist() == [0, 2]
    c4, o4 = _fm_patterns([])
    assert c4.size == 0 and o4.tolist() == [0]
