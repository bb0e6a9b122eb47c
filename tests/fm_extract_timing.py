"""Timing of extract on the device (grlgpu_fm_extract), one JSON line per workload.

Each workload is built with build_bwt_packed in the same command and loaded with fm_load. Timed, by CUDA events on the context's
stream: device_ms (request upload, extraction, result download) and extract_ms (the extraction alone) of one call; one warm-up,
then the median of `--reps`.
- reads, dna_reads(8e6, 150): 10^6 whole reads at random k (length None: GrlGpu.fm_extract sizes the output by a first call
  without capacity, and the times are those of both calls) and 10^6 windows of 32, on the automatic choice (the walk), then both
  with GRLGPU_FLAG_FORCE_JUMP, where the first call after a load builds the locate table and the samples and the second reuses them.
- long, repetitive_genomes(100, 4e6): 10^5 windows of 32 and 100 windows of 10^5, each as the first call after a load (the count
  pass gives up at the bound, the table and the samples are built) and as a second call; and 10^3 windows of 32 with
  GRLGPU_FLAG_FORCE_WALK, every request walking from its string's end.
The host tool fm_extract answers the first 10^4 windows of 32 (wall clock of the process, .rl_bwt reading included) and its output
must equal fm_extract_gpu's. The GPU name and power limit are read by nvidia-smi in the same command.

    python tests/fm_extract_timing.py [--out profiles/r04_fm_extract_timing.jsonl] [--only reads,long] [--reps 3]
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
N_HOST = 10_000


def windows(arr, rng, n_req, m):
    """n_req windows of m symbols inside the strings at least m long -> (k, from, len)"""
    sep = arr[-1]
    ends = np.flatnonzero(arr == sep)
    starts = np.concatenate(([0], ends[:-1] + 1))
    ok = np.flatnonzero(ends - starts >= m)
    k = rng.choice(ok, n_req)
    f = (rng.random(n_req) * (ends[k] - starts[k] - m + 1)).astype(np.int64)
    return k, f, np.full(n_req, m, np.int64)


def summary(runs):
    med = lambda key: round(float(np.median([r[key] for r in runs])), 3)  # noqa: E731
    d = runs[-1]
    return {"path": ["walk", "samples"][d["path"]], "n_req": d["n_req"], "n_cells": d["n_cells"], "jump_rounds": d["jump_rounds"],
            "device_ms": med("device_ms"), "extract_ms": med("extract_ms"), "cells_per_s": round(d["n_cells"] / med("device_ms") * 1e3)}


def steady(ctx, req, reps):
    """one warm-up, then `reps` calls"""
    ctx.fm_extract(*req)
    return summary([ctx.fm_extract(*req)[2] for _ in range(reps)])


def first_second(ctx, img, req, reps):
    """the first call after a load and the second call, each `reps` times after one warm-up round"""
    firsts, seconds = [], []
    for _ in range(reps + 1):
        ctx.fm_load(img)
        firsts.append(ctx.fm_extract(*req)[2])
        seconds.append(ctx.fm_extract(*req)[2])
    return {"first_call": summary(firsts[1:]), "second_call": summary(seconds[1:])}


def host_check(img, req, tmp):
    rl, rq, ho, do = (os.path.join(tmp, x) for x in ("x.rl_bwt", "req.txt", "host.bin", "dev.bin"))
    img.tofile(rl)
    k, f, m = req
    with open(rq, "w") as fh:
        fh.write("".join(f"{a} {b} {c}\n" for a, b, c in zip(k.tolist(), f.tolist(), m.tolist())))
    t0 = time.perf_counter()
    h = subprocess.run([os.path.join(G.LIB_DIR, "fm_extract"), rl, rq, ho], capture_output=True)
    host_s = time.perf_counter() - t0
    assert h.returncode == 0, h.stderr
    t0 = time.perf_counter()
    d = subprocess.run([os.path.join(G.LIB_DIR, "fm_extract_gpu"), rl, rq, do], capture_output=True)
    tool_s = time.perf_counter() - t0
    assert d.returncode == 0, d.stderr
    with open(ho, "rb") as a, open(do, "rb") as b:
        equal = a.read() == b.read()
    return {"host_n_req": int(k.size), "host_fm_extract_s": round(host_s, 3), "fm_extract_gpu_s": round(tool_s, 3), "host_output_equal": equal}


def check(arr, req, off, cells):
    """the cells of every request against numpy slices of the collection"""
    sep = arr[-1]
    ends = np.flatnonzero(arr == sep)
    starts = np.concatenate(([0], ends[:-1] + 1))
    k, f, m = req
    lo = starts[k] + f
    cnt = np.maximum(np.minimum(lo + m, ends[k]) - lo, 0)
    idx = np.repeat(lo - np.concatenate(([0], np.cumsum(cnt)[:-1])), cnt) + np.arange(int(cnt.sum()))
    return bool(np.array_equal(np.diff(off.astype(np.int64)), cnt) and np.array_equal(cells, arr[idx]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_fm_extract_timing.jsonl"))
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
        res = {"workload": name, "gpu": card, "n": int(arr.size), "n_runs": n_runs, "image_bytes": nb, "B": max(4096, arr.size // 2048),
               "sample_rate": 64}
        w32 = windows(arr, rng, 1_000_000 if name == "reads" else 100_000, 32)
        with G.GrlGpu(0) as ctx:
            res["n_strings"] = ctx.fm_load(img)["n_strings"]
            if name == "reads":
                whole = (rng.integers(0, res["n_strings"], 1_000_000), 0, None)
                res["whole_reads"] = steady(ctx, whole, a.reps)
                res["windows32"] = steady(ctx, w32, a.reps)
                off, cells, _ = ctx.fm_extract(*w32)
                res["windows32"]["equal_numpy"] = check(arr, w32, off, cells)
            else:
                w1e5 = windows(arr, rng, 100, 100_000)
                res["windows32"] = first_second(ctx, img, w32, a.reps)
                res["windows1e5"] = first_second(ctx, img, w1e5, a.reps)
                for key, req in (("windows32", w32), ("windows1e5", w1e5)):
                    off, cells, _ = ctx.fm_extract(*req)
                    res[key]["equal_numpy"] = check(arr, req, off, cells)
        if name == "reads":
            with G.GrlGpu(0, G.FLAG_FORCE_JUMP) as ctx:
                res["whole_reads_jump"] = first_second(ctx, img, whole, a.reps)
                res["windows32_jump"] = first_second(ctx, img, w32, a.reps)
        else:
            walk = tuple(x[:1000] for x in w32)
            with G.GrlGpu(0, G.FLAG_FORCE_WALK) as ctx:
                ctx.fm_load(img)
                res["windows32_walk_1e3"] = steady(ctx, walk, a.reps)
        with tempfile.TemporaryDirectory() as tmp:
            res.update(host_check(img, tuple(x[:N_HOST] for x in w32), tmp))
        print(json.dumps(res), flush=True)
        lines.append(json.dumps(res))
        del arr, img
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
