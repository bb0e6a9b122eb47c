"""Timing of the LCP array on the device (grlgpu_fm_lcp), one JSON line per workload.

Each workload is built with build_bwt_packed in the same command and loaded with fm_load. Timed, by CUDA events on the context's
stream: device_ms (the whole call, with the download of the 4·n-byte array into pageable memory), sa_ms (SA and the text) and
lcp_ms (irreducible rows, their comparisons, the max-scan and the gather) of one call, on the automatic choice and under
GRLGPU_FLAG_FORCE_WALK and GRLGPU_FLAG_FORCE_JUMP, each in a fresh context: the first call after the load (which builds the locate
table on the table path) is the warm-up and is recorded apart, then the median of `--reps` calls.
- reads, dna_reads(8e6, 150): strings of 150, the walk per string.
- long, repetitive_genomes(100, 4e6): strings of 4·10⁶, longer than the walk bound, so the table; long comparisons.
The three paths must give the same array. The host tool fm_lcp runs on a prefix of each collection (whole strings, about 10⁷
symbols; wall clock of the process, .rl_bwt reading included), and its output must equal the device's on that prefix. The GPU
name and power limit are read by nvidia-smi in the same command.

    python tests/fm_lcp_timing.py [--out profiles/r06_fm_lcp_timing.jsonl] [--only reads,long] [--reps 3]
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
import gen  # noqa: E402
import grlbwt_b200 as G  # noqa: E402
from invert_timing import gpu_card  # noqa: E402

WORKLOADS = {
    "reads": lambda: gen.dna_reads(8_000_000, 150, seed=42),
    "long": lambda: gen.repetitive_genomes(100, 4_000_000, seed=7),
}
HOST_PREFIX = 10_000_000   # symbols of the prefix the host tool answers (whole strings)
FLAGS = {"auto": 0, "walk": G.FLAG_FORCE_WALK, "jump": G.FLAG_FORCE_JUMP}


def image(arr):
    img = np.empty(16 + arr.size * 16, np.uint8)
    nb, n_runs, _, _, _ = G.build_bwt_packed(arr, img, n_threads=16)
    return img[:nb].copy(), n_runs


def summary(runs):
    med = lambda key: round(float(np.median([r[key] for r in runs])), 3)  # noqa: E731
    d = runs[-1]
    return {"path": ["walk", "table"][d["path"]], "device_ms": med("device_ms"), "sa_ms": med("sa_ms"), "lcp_ms": med("lcp_ms"),
            "n_irreducible": d["n_irreducible"], "sum_irreducible": d["sum_irreducible"],
            "rows_per_s": round(d["n"] / med("device_ms") * 1e3)}


def time_flags(img, flags, reps):
    """the first call after a load, then `reps` calls -> (record, last array)"""
    with G.GrlGpu(0, flags) as ctx:
        ctx.fm_load(img)
        lcp, first = ctx.fm_lcp()
        runs = []
        for _ in range(reps):
            lcp, info = ctx.fm_lcp()
            runs.append(info)
    rec = summary(runs)
    rec["first_call"] = {"device_ms": round(first["device_ms"], 3), "sa_ms": round(first["sa_ms"], 3), "jump_rounds": first["jump_rounds"]}
    return rec, lcp


def host_check(arr, tmp):
    """the host tool on a prefix of whole strings against the device on the same prefix"""
    ends = np.flatnonzero(arr == arr[-1])
    cut = int(ends[max(np.searchsorted(ends, HOST_PREFIX) - 1, 0)]) + 1
    img, _ = image(arr[:cut])
    rl, ho = os.path.join(tmp, "p.rl_bwt"), os.path.join(tmp, "host.bin")
    img.tofile(rl)
    t0 = time.perf_counter()
    h = subprocess.run([os.path.join(G.LIB_DIR, "fm_lcp"), rl, ho], capture_output=True)
    host_s = time.perf_counter() - t0
    assert h.returncode == 0, h.stderr
    with G.GrlGpu(0) as ctx:
        ctx.fm_load(img)
        ctx.fm_lcp()
        dev, info = ctx.fm_lcp()
    return {"host_prefix_n": cut, "host_fm_lcp_s": round(host_s, 3), "device_prefix_ms": round(info["device_ms"], 3),
            "host_output_equal": bool(np.array_equal(np.fromfile(ho, "<u4"), dev))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_fm_lcp_timing.jsonl"))
    ap.add_argument("--only", default=",".join(WORKLOADS))
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    card = gpu_card()
    lines = []
    for name in a.only.split(","):
        arr = WORKLOADS[name]()
        img, n_runs = image(arr)
        res = {"workload": name, "gpu": card, "n": int(arr.size), "n_runs": n_runs, "image_bytes": int(img.size), "B": max(4096, arr.size // 2048)}
        ref = None
        equal = True
        for key, flags in FLAGS.items():
            res[key], lcp = time_flags(img, flags, a.reps)
            if ref is None:
                ref = lcp
            else:
                equal = equal and bool(np.array_equal(lcp, ref))
            del lcp
        res["paths_equal"] = equal
        res["max_lcp"] = int(ref.max())
        del ref
        with tempfile.TemporaryDirectory() as tmp:
            res.update(host_check(arr, tmp))
        print(json.dumps(res), flush=True)
        lines.append(json.dumps(res))
        del arr, img
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
