"""CPU suite: the host extract tool fm_extract against numpy slices of the collections and against reverse_bwt, both tools' usage,
the requests-file rules and the argument checks of GrlGpu.fm_extract (no device needed)."""
import subprocess

import numpy as np
import pytest

import gen
import grlbwt_b200 as G
from extract_oracle import U32_MAX, low_bytes, requests, requests_file, tool_output
from fm_oracle import Text, image_of, lib
from grlbwt_b200.api import _fm_requests


def run_extract(rl, req_path, out_path, w):
    r = subprocess.run([lib("fm_extract"), str(rl), str(req_path), str(out_path), "-a", str(w)], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    return out_path.read_bytes()


def check_case(arr, tmp_path, seed):
    raw, _ = image_of(arr)
    rl, rq, out = tmp_path / "x.rl_bwt", tmp_path / "req.txt", tmp_path / "out.bin"
    rl.write_bytes(raw)
    t, w = Text(arr), arr.dtype.itemsize
    reqs = requests(t, np.random.default_rng(seed))
    requests_file(rq, reqs)
    assert run_extract(rl, rq, out, w) == tool_output(t, reqs, w)


@pytest.mark.parametrize("name", list(gen.small_cases()))
def test_fm_extract_small_cases(name, tmp_path):
    check_case(gen.small_cases()[name], tmp_path, 3)


def test_fm_extract_fuzz(tmp_path):
    for i, (name, arr) in enumerate(gen.fuzz_cases()):
        check_case(arr, tmp_path, i)


@pytest.mark.parametrize("name", ["with_empty", "dna_500", "u16_small_sigma", "u32_small_sigma", "u64_rand", "high_bytes", "fuzz"])
def test_all_strings_equal_reverse_bwt(name, tmp_path):
    """requests 0 .. N-1 without from or len write what reverse_bwt writes, at every cell width (the low bytes where symbols do
    not fit)"""
    arr = dict(gen.fuzz_cases())["fuzz_0"] if name == "fuzz" else gen.small_cases()[name]
    raw, _ = image_of(arr)
    rl, rq, out, rev = tmp_path / "x.rl_bwt", tmp_path / "req.txt", tmp_path / "out.bin", tmp_path / "rev.bin"
    rl.write_bytes(raw)
    t = Text(arr)
    rq.write_text("".join(f"{k}\n" for k in range(t.ends.size)))
    for w in (1, 2, 4, 8):
        got = run_extract(rl, rq, out, w)
        r = subprocess.run([lib("reverse_bwt"), str(rl), str(rev), "-a", str(w)], capture_output=True)
        assert r.returncode == 0, r.stderr.decode()
        assert got == rev.read_bytes() == low_bytes(arr, w).tobytes(), (name, w)


@pytest.mark.parametrize("tool", ["fm_extract", "fm_extract_gpu"])
def test_usage(tool):
    r = subprocess.run([lib(tool)], capture_output=True, text=True)
    assert r.returncode == 0 and "usage:" in r.stdout


@pytest.mark.parametrize("text,msg", [
    ("1 2 3 4\n", "line 1"),            # four fields
    ("0\nx\n", "line 2"),               # not a number
    ("0\n-1\n", "line 2"),              # negative
    ("0 1,2\n", "line 1"),              # another separator
    ("0\n\n1\n", "line 2"),             # an empty line
    ("0 2x\n", "line 1"),               # trailing garbage
    ("0 18446744073709551616\n", "line 1"),   # beyond 64 bits
    ("0\n7\n", "does not exist"),       # k = N
    ("99999999999\n", "does not exist"),
])
def test_request_file_errors(tmp_path, text, msg):
    arr = gen.small_cases()["with_empty"]   # N = 7
    assert Text(arr).ends.size == 7
    raw, _ = image_of(arr)
    rl, rq, out = tmp_path / "x.rl_bwt", tmp_path / "req.txt", tmp_path / "out.bin"
    rl.write_bytes(raw)
    rq.write_text(text)
    r = subprocess.run([lib("fm_extract"), str(rl), str(rq), str(out)], capture_output=True, text=True)
    assert r.returncode == 1 and "Error:" in r.stderr and msg in r.stderr, r.stderr


def test_request_file_forms(tmp_path):
    """"k", "k from", "k from len", blanks and tabs between fields, a last line without newline, len beyond the string"""
    arr = gen.small_cases()["with_empty"]
    raw, _ = image_of(arr)
    t = Text(arr)
    rl, rq, out = tmp_path / "x.rl_bwt", tmp_path / "req.txt", tmp_path / "out.bin"
    rl.write_bytes(raw)
    rq.write_text("0\n 1  2\n2\t1\t3\n3 0 18446744073709551615")
    want = tool_output(t, [(0, None, None), (1, 2, None), (2, 1, 3), (3, 0, None)], 1)
    assert run_extract(rl, rq, out, 1) == want


@pytest.mark.parametrize("args", [
    dict(str_id=-1),                              # negative
    dict(str_id=[0, 1], start=[0, -3]),
    dict(str_id=[0, 1], length=-1),
    dict(str_id=[1 << 32]),                       # str_id beyond 32 bits
    dict(str_id=[0, 1], start=[0, 1, 2]),         # mismatched lengths
    dict(str_id=[0, 1, 2], length=[5, 6]),
    dict(str_id=0, cell_bytes=3),                 # bad cell_bytes
    dict(str_id=0, cell_bytes=16),
    dict(str_id=[0.5]),                           # not integers
    dict(str_id=[[0, 1]]),                        # not 1-d
])
def test_request_argument_checks(args):
    with pytest.raises(G.GrlGpuError) as e:
        _fm_requests(**args)
    assert e.value.status == -1


def test_request_forms():
    ids, frm, ln = _fm_requests([3, 1, 2], 5, None)
    assert [a.dtype for a in (ids, frm, ln)] == [np.uint32] * 3 and all(a.flags["C_CONTIGUOUS"] for a in (ids, frm, ln))
    assert ids.tolist() == [3, 1, 2] and frm.tolist() == [5, 5, 5] and ln.tolist() == [U32_MAX] * 3
    ids, frm, ln = _fm_requests(np.array([7], np.int64), [1 << 40], [1 << 33])   # a start beyond 32 bits is empty
    assert ids.tolist() == [7] and frm.tolist() == [U32_MAX] and ln.tolist() == [0]
    ids, frm, ln = _fm_requests([7, 8], 2, [1 << 33, 4])                           # a length beyond 32 bits runs to the end
    assert frm.tolist() == [2, 2] and ln.tolist() == [U32_MAX, 4]
    ids, frm, ln = _fm_requests(9)
    assert ids.tolist() == [9] and frm.tolist() == [0] and ln.tolist() == [U32_MAX]
    assert all(a.size == 0 for a in _fm_requests([]))
