"""Timing of the search with mismatches on the device (grlgpu_fm_approx_count / _locate), one JSON line per workload.

The workloads of tests/fm_timing.py, each built with build_bwt_packed in the same command. Pattern sets: 10^5 windows of 32 and of
150 sampled from the strings, each with 0, 1 or 2 random substitutions, and 10^5 random patterns of 32. Runs: k = 1, 2, 3 on the
length-32 sets, k = 1, 2 on the length-150 set. Per run, by CUDA events on the context's stream: device_ms (whole count call:
pattern upload, search, sort, result download), search_ms, n_hits, n_occ, n_lf and LF_c evaluations per second of search; then
locate on the first 10^4 patterns (device_ms, locate_ms, path; on the long genomes the first locate builds the locate table, so
it is warmed up before). One warm-up, then the median of `--reps`. The host tool fm_query -k 2 answers the first 10^3 patterns of
the sampled length-32 set (with -l on the reads; counts only on the long genomes, where each host locate walks millions of LF
steps) and its output must equal fm_query_gpu's bytes. The GPU name and power limit are read by nvidia-smi in the same command.

    python tests/fm_approx_timing.py [--out profiles/r05_fm_approx_timing.jsonl] [--only reads,long] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import grlbwt_b200 as G  # noqa: E402
from approx_oracle import mutate  # noqa: E402
from fm_timing import WORKLOADS, median_of, sample  # noqa: E402
from invert_timing import gpu_card  # noqa: E402

N_PAT, N_LOC, N_HOST = 100_000, 10_000, 1_000
DNA = np.frombuffer(b"ACGT", np.uint8)


def mutated(arr, rng, m):
    cells, off = sample(arr, rng, N_PAT, m)
    return mutate(rng, cells.reshape(N_PAT, m), DNA, rng.integers(0, 3, N_PAT)).ravel(), off


def host_check(img, arr, cells, off, tmp, locate, kmax):
    sep = int(arr[-1])
    rl, pp = os.path.join(tmp, "x.rl_bwt"), os.path.join(tmp, "p.bin")
    img.tofile(rl)
    n = off.size - 1
    with open(pp, "wb") as f:
        f.write(np.insert(cells.reshape(n, -1), cells.size // n, sep, axis=1).astype(arr.dtype).tobytes())
    cmd = [rl, pp, "-k", str(kmax)] + (["-l"] if locate else [])
    t0 = time.perf_counter()
    h = subprocess.run([os.path.join(G.LIB_DIR, "fm_query")] + cmd, capture_output=True)
    host_s = time.perf_counter() - t0
    assert h.returncode == 0, h.stderr
    t0 = time.perf_counter()
    d = subprocess.run([os.path.join(G.LIB_DIR, "fm_query_gpu")] + cmd, capture_output=True)
    tool_s = time.perf_counter() - t0
    assert d.returncode == 0, d.stderr
    return {"host_n_pat": n, "host_k": kmax, "host_locate": locate, "host_fm_query_s": round(host_s, 3), "fm_query_gpu_s": round(tool_s, 3),
            "host_output_equal": h.stdout == d.stdout}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_fm_approx_timing.jsonl"))
    ap.add_argument("--only", default=",".join(WORKLOADS))
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    card = gpu_card()
    lines = []
    for name in a.only.split(","):
        arr = WORKLOADS[name]()
        img = np.empty(16 + arr.size * 16, np.uint8)
        nb, n_runs, _, _, _ = G.build_bwt_packed(arr, img, n_threads=16)
        img = img[:nb].copy()
        rng = np.random.default_rng(1)
        sets = {"sampled32": mutated(arr, rng, 32), "random32": (rng.choice(DNA, N_PAT * 32), np.arange(0, N_PAT * 32 + 1, 32, dtype=np.uint64)),
                "sampled150": mutated(arr, rng, 150)}
        res = {"workload": name, "gpu": card, "n": int(arr.size), "n_runs": n_runs, "runs": []}
        with G.GrlGpu(0) as ctx:
            info = ctx.fm_load(img)
            res["sigma"], res["n_strings"] = info["sigma"], info["n_strings"]
            for key, ks in (("sampled32", (1, 2, 3)), ("random32", (1, 2, 3)), ("sampled150", (1, 2))):
                cells, off = sets[key]
                m = int(off[1])
                loc = (cells[:N_LOC * m], off[:N_LOC + 1])
                for kmax in ks:
                    runs, med = median_of(lambda: ctx.fm_approx_count((cells, off), kmax)[4], a.reps)
                    search = float(np.median([r["search_ms"] for r in runs]))
                    lruns, lmed = median_of(lambda: ctx.fm_approx_locate(loc, kmax)[4], a.reps)
                    r = runs[-1]
                    res["runs"].append({"set": key, "m": m, "k": kmax, "n_pat": N_PAT, "device_ms": round(med, 3), "search_ms": round(search, 3),
                                        "n_hits": r["n_hits"], "n_occ": r["n_occ"], "n_lf": r["n_lf"], "lf_per_s": round(r["n_lf"] / search * 1e3),
                                        "locate_n_pat": N_LOC, "locate_device_ms": round(lmed, 3),
                                        "locate_ms": round(float(np.median([x["locate_ms"] for x in lruns])), 3),
                                        "locate_path": ["walk", "table"][lruns[-1]["path"]], "locate_n_occ": lruns[-1]["n_occ"]})
                    print(json.dumps(res["runs"][-1]), flush=True)
        cells, off = sets["sampled32"]
        with tempfile.TemporaryDirectory() as tmp:
            res.update(host_check(img, arr, cells[:N_HOST * 32], off[:N_HOST + 1], tmp, name == "reads", 2))
        print(json.dumps(res), flush=True)
        lines.append(json.dumps(res))
        del arr, img
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
