"""Generate tests/golden/tools_golden.json: what the .rl_bwt consumer scripts of the reference (scripts/grl2plain.cpp,
grlbwt2rle.cpp, bwt_stats.cpp, split_runs.cpp) produce on the .rl_bwt files of a few seeded cases, as sha256 of the output
files and the lines of the bwt_stats report. tests/test_tools_cpu.py compares grlbwt_b200/host/tools with these values.

The values are recorded from grlbwt_b200/host/tools, which were checked byte for byte against the reference's own scripts
on the same inputs when those were built alongside (split_runs: the reference's output minus the zero-length records it
emits when a run ends exactly on a block boundary). The reference itself is not part of this repository.
    make -C grlbwt_b200 && python tests/golden/make_tools_golden.py
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import gen  # noqa: E402
import grlbwt_b200 as G  # noqa: E402
from oracle import oracle as O  # noqa: E402

PLAIN_CASES = ["rep_50x200k", "mixed_reads", "homopolymers_multi", "test_byte_alphabet"]
SPLIT_CASES = ["rep_50x200k", "homopolymers_multi", "mixed_reads"]
# (bits, block size) of tests/test_tools_cpu.py::test_split_runs that the reference handles (block size >= 64; the last
# block size, one more than the BWT length, is filled in per case)
SPLIT_CONFIGS = [(3, 1000), (2, 64), (8, 4096), (5, 999983), (4, None)]


def sha(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def run(*cmd):
    r = subprocess.run([str(c) for c in cmd], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"{cmd[0]}: {r.stderr}")
    return r.stdout


def bwt_report(stdout):
    """the lines of the reference's report (tools/bwt_stats.cpp prints a summary of the file after a blank line)"""
    lines = stdout.splitlines()
    return lines[: lines.index("")] if "" in lines else lines


def rl_bwt_file(arr, path):
    o = O.Oracle(arr)
    o.par_phase()
    syms, lens, sb, fb = o.ind_phase()
    o.close()
    with open(path, "wb") as f:
        f.write(O.rl_bwt_bytes(syms, lens, sb, fb))
    return len(syms), int(lens.sum())


def main():
    cases = {"test_byte_alphabet": gen.fixture_byte_alphabet()}
    cases.update(gen.small_cases())
    cases["rep_50x200k"] = gen.repetitive_genomes(50, 200000, seed=7)
    cases["mixed_reads"] = gen.mixed_reads(20000, 30, 150, 10000, seed=5)
    tool = lambda name: os.path.join(G.LIB_DIR, name)  # noqa: E731
    out = {"generator": "tests/golden/make_tools_golden.py", "cases": {}}
    with tempfile.TemporaryDirectory() as td:
        for name in sorted(set(PLAIN_CASES) | set(SPLIT_CASES)):
            rl = os.path.join(td, name + ".rl_bwt")
            n_runs, n_syms = rl_bwt_file(cases[name], rl)
            rec = out["cases"][name] = {"rl_bwt_sha256": sha(rl)}
            if name in PLAIN_CASES:
                p = os.path.join(td, "plain")
                run(tool("grl2plain"), rl, p)
                rec["grl2plain_sha256"] = sha(p)
                run(tool("grlbwt2rle"), rl, p)
                rec["grlbwt2rle_syms_sha256"], rec["grlbwt2rle_len_sha256"] = sha(p + ".syms"), sha(p + ".len")
                if n_runs >= 20:   # the reference reads one past its sorted lengths when there are fewer than 10 runs
                    rec["bwt_stats_report"] = bwt_report(run(tool("bwt_stats"), rl))
            if name in SPLIT_CASES:
                rec["split_runs"] = {}
                for bits, n in SPLIT_CONFIGS:
                    n = n or n_syms + 1
                    s = os.path.join(td, f"s_{bits}_{n}")
                    run(tool("split_runs"), rl, bits, n, s)
                    rec["split_runs"][f"{bits}_{n}"] = {"sha256": sha(s), "dist_sha256": sha(s + ".dist")}
            print(name, rec["rl_bwt_sha256"][:16], flush=True)
    with open(os.path.join(HERE, "tools_golden.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
