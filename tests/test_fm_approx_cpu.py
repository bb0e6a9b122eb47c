"""CPU suite: the host search with mismatches (fm_query -k) against every window of the collections, -k 0 against the exact
search, the tools' -k range, and the argument checks of GrlGpu.fm_approx_count / fm_approx_locate (no device needed)."""
import subprocess

import numpy as np
import pytest

import gen
import grlbwt_b200 as G
from approx_oracle import naive, parse_output, patterns
from fm_oracle import Text, image_of, lib, patterns_file
from grlbwt_b200.api import _fm_approx_args


def run_k(rl, pp, w, kmax, locate, tool="fm_query"):
    cmd = [lib(tool), str(rl), str(pp), "-a", str(w), "-k", str(kmax)] + (["-l"] if locate else [])
    r = subprocess.run(cmd, capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    return r.stdout


def check_host_tool(arr, tmp_path, seed):
    raw, _ = image_of(arr)
    rl, pp = tmp_path / "x.rl_bwt", tmp_path / "p.bin"
    rl.write_bytes(raw)
    t, w = Text(arr), arr.dtype.itemsize
    pats = [p for p in patterns(t, np.random.default_rng(seed)) if t.sep not in p]
    patterns_file(pp, pats, t.sep, w)
    exact = subprocess.run([lib("fm_query"), str(rl), str(pp), "-a", str(w)], capture_output=True).stdout
    assert run_k(rl, pp, w, 0, False) == exact
    longest = int((t.ends - t.starts).max()) + 1
    for kmax in (0, 1, 2):
        want = [naive(t, p, kmax) for p in pats]
        counts = parse_output(run_k(rl, pp, w, kmax, False))
        assert [c for c, _ in counts] == [len(x) for x in want], kmax
        if kmax == 0:
            continue   # -k 0 with -l is the exact search's output, checked by the fm_query suite
        small = [q for q in range(len(pats)) if len(want[q]) * longest <= 2_000_000]
        patterns_file(pp, [pats[q] for q in small], t.sep, w)
        got = parse_output(run_k(rl, pp, w, kmax, True))
        patterns_file(pp, pats, t.sep, w)
        assert len(got) == len(small)
        for q, (cnt, occ) in zip(small, got):
            assert cnt == len(want[q]) and sorted(occ) == want[q], (kmax, pats[q])


@pytest.mark.parametrize("name", list(gen.small_cases()))
def test_fm_query_k_small_cases(name, tmp_path):
    check_host_tool(gen.small_cases()[name], tmp_path, 7)


def test_fm_query_k_fuzz(tmp_path):
    for i, (name, arr) in enumerate(gen.fuzz_cases()):
        check_host_tool(arr, tmp_path, i)


def test_k0_is_the_exact_search(tmp_path):
    arr = gen.small_cases()["dna_500"]
    raw, _ = image_of(arr)
    rl, pp = tmp_path / "x.rl_bwt", tmp_path / "p.bin"
    rl.write_bytes(raw)
    t = Text(arr)
    patterns_file(pp, t.patterns(np.random.default_rng(2)), t.sep, 1)
    for loc in ([], ["-l"]):
        plain = subprocess.run([lib("fm_query"), str(rl), str(pp)] + loc, capture_output=True)
        with_k = subprocess.run([lib("fm_query"), str(rl), str(pp), "-k", "0"] + loc, capture_output=True)
        assert plain.returncode == with_k.returncode == 0 and plain.stdout == with_k.stdout


@pytest.mark.parametrize("tool", ["fm_query", "fm_query_gpu"])
def test_usage_and_k_range(tool, tmp_path):
    r = subprocess.run([lib(tool)], capture_output=True, text=True)
    assert r.returncode == 0 and "-k" in r.stdout
    arr = gen.small_cases()["with_empty"]
    raw, _ = image_of(arr)
    rl, pp = tmp_path / "x.rl_bwt", tmp_path / "p.bin"
    rl.write_bytes(raw)
    pp.write_bytes(b"AC\n")
    for bad in ("4", "-1", "x", "12"):
        r = subprocess.run([lib(tool), str(rl), str(pp), "-k", bad], capture_output=True, text=True)
        assert r.returncode == 1 and "-k" in r.stderr, (bad, r.stderr)


@pytest.mark.parametrize("k", [-1, 4, 1.5, "1", None])
def test_k_argument_checks(k):
    with pytest.raises(G.GrlGpuError) as e:
        _fm_approx_args([b"AC"], k)
    assert e.value.status == -1


def test_approx_pattern_checks():
    with pytest.raises(G.GrlGpuError):
        _fm_approx_args([b"AC", b""], 1)
    cells, off, k = _fm_approx_args((np.frombuffer(b"ACGT", np.uint8), np.array([0, 1, 4])), np.uint8(2))
    assert k == 2 and off.tolist() == [0, 1, 4] and cells.dtype == np.uint8
