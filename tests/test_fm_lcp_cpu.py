"""CPU suite: the host LCP tool fm_lcp against the oracle of lcp_oracle.py on every small and fuzz case at 1-, 2- and 4-byte
alphabets, the oracle's row order against the collection, and the usage and error exits of both tools (no device needed)."""
import subprocess

import numpy as np
import pytest

import gen
from fm_oracle import image_of, lib
from lcp_oracle import check_order, lcp_of


def run_lcp(raw, tmp_path):
    rl, out = tmp_path / "x.rl_bwt", tmp_path / "lcp.bin"
    rl.write_bytes(raw)
    r = subprocess.run([lib("fm_lcp"), str(rl), str(out)], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    return np.fromfile(out, "<u4")


def check_case(arr, tmp_path):
    raw, _ = image_of(arr)
    want, rows, pos = lcp_of(arr, raw)
    check_order(arr, want, pos, rows.sep)
    got = run_lcp(raw, tmp_path)
    assert got.size == rows.n and np.array_equal(got, want)
    assert (got[:rows.N] == 0).all()


def widened(arr, dtype, base):
    """the same collection over a wider alphabet: every symbol moved up by `base`, so the order and the LCP stay"""
    return arr.astype(dtype) + dtype(base)


@pytest.mark.parametrize("name", list(gen.small_cases()))
def test_fm_lcp_small_cases(name, tmp_path):
    check_case(gen.small_cases()[name], tmp_path)


@pytest.mark.parametrize("dtype,base", [(np.uint8, 0), (np.uint16, 1000), (np.uint32, 70000)])
def test_fm_lcp_fuzz(dtype, base, tmp_path):
    for name, arr in gen.fuzz_cases():
        check_case(widened(arr, dtype, base), tmp_path)


@pytest.mark.parametrize("tool", ["fm_lcp", "fm_lcp_gpu"])
def test_usage(tool):
    r = subprocess.run([lib(tool)], capture_output=True, text=True)
    assert r.returncode == 0 and "usage:" in r.stdout


def image_of_runs(syms, lens, sb=4, fb=4):
    from oracle import oracle as O
    return O.rl_bwt_bytes(np.asarray(syms, np.uint64), np.asarray(lens, np.uint64), sb, fb)


@pytest.mark.parametrize("image", [
    b"",                                                          # no header
    np.array([3, 0], np.uint64).tobytes(),                        # fb = 0
    np.array([1, 1], np.uint64).tobytes() + b"\x01",              # a truncated record
    "run list 1 3 2",                                             # LF cycles without separator
    "run list 1 4 2 3",
    "run list 1 2 1 4 3 5",
])
def test_malformed_images(image, tmp_path):
    if isinstance(image, str):
        from oracle import oracle as O
        s, lens = O.rle(np.array([int(x) for x in image.split()[2:]]))
        image = image_of_runs(s, lens)
    rl, out = tmp_path / "x.rl_bwt", tmp_path / "lcp.bin"
    rl.write_bytes(image)
    r = subprocess.run([lib("fm_lcp"), str(rl), str(out)], capture_output=True, text=True)
    assert r.returncode == 1 and "Error:" in r.stderr, (r.returncode, r.stderr)


def test_missing_file(tmp_path):
    r = subprocess.run([lib("fm_lcp"), str(tmp_path / "none.rl_bwt"), str(tmp_path / "o")], capture_output=True, text=True)
    assert r.returncode == 1 and "Error:" in r.stderr
