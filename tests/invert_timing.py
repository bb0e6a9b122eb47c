"""Timing of the device inversion (grlgpu_invert), one JSON line per workload.

Every workload is built with build_bwt_packed in the same command, then inverted automatically and with each path forced
(GRLGPU_FLAG_FORCE_WALK / _JUMP), so that both sides of the selection are measured on it: one warm-up call, then the median of
`--reps` calls by device_ms (CUDA events around the whole call: image upload, LF table, inversion, output download; image and
output are in pinned memory). Each output is checked against the text. The walk on the single-string workload is not timed by default: it is one
chain of n dependent loads (--walk-one-string times it). Reported per path: MB/s as n * w / device_ms, lf_ms and invert_ms, the
path and jump rounds, and the inversion's achieved bytes/s against the traffic model below. The host tool reverse_bwt is timed
on the first `host_k` strings (wall clock of the process, LF structure built from the file included) against the device
inversion of the same strings. The GPU name and power limit are read by nvidia-smi in the same command.

    python tests/invert_timing.py [--only reads,mixed,long,one] [--reps 3]
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

# name -> (generator, strings the host tool inverts)
WORKLOADS = {
    "reads": (lambda: gen.dna_reads(8_000_000, 150, seed=42), 100_000),
    "mixed": (lambda: gen.mixed_reads(200_000, 300, 150, 10_000, seed=5), 100_000),
    "long": (lambda: gen.repetitive_genomes(100, 4_000_000, seed=7), 1),
    "one": (lambda: gen.repetitive_genomes(1, 256_000_000 - 1, seed=9), 0),
}


def model_bytes(info, w):
    """DRAM bytes the inversion needs: walk: two passes of one 32 B sector per LF step, plus the output; jumping: per round and
    entry 8 B read + one 32 B sector gathered + 8 B written"""
    steps = info["n_out"] - min(info["n_strings"], info["n_out"])
    if info["path"] == 0:
        return 2 * 32 * steps + info["n_out"] * w
    return info["jump_rounds"] * info["n"] * (8 + 32 + 8)


def gpu_card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def pinned(nbytes):
    import torch
    return torch.empty(max(nbytes, 1), dtype=torch.uint8, pin_memory=True).numpy()


def time_path(img, arr, flags, reps, out):
    w = arr.dtype.itemsize
    with G.GrlGpu(0, flags) as ctx:
        got, info = ctx.invert(img, w, out=out)   # warm-up
        ok = got.size == arr.size and np.array_equal(got, arr)
        ms = []
        for _ in range(reps):
            got, info = ctx.invert(img, w, out=out)
            ok = ok and np.array_equal(got, arr)
            ms.append(info["device_ms"])
    med = float(np.median(ms))
    mb = model_bytes(info, w)
    return {"path": ["walk", "jump"][info["path"]], "jump_rounds": info["jump_rounds"], "device_ms": round(med, 3),
            "device_ms_all": [round(x, 3) for x in ms], "lf_ms": round(info["lf_ms"], 3), "invert_ms": round(info["invert_ms"], 3),
            "MB_per_s": round(arr.size * w / med / 1e3, 1), "model_bytes": mb, "achieved_GB_per_s": round(mb / info["invert_ms"] / 1e6, 1),
            "output_equals_text": bool(ok)}


def host_vs_device(img, arr, k, tmp):
    if k == 0:
        return {"host_reverse_bwt": "not measured"}
    w = arr.dtype.itemsize
    rl, out = os.path.join(tmp, "x.rl_bwt"), os.path.join(tmp, "x.out")
    img.tofile(rl)
    t0 = time.perf_counter()
    r = subprocess.run([os.path.join(G.LIB_DIR, "reverse_bwt"), rl, out, str(k), "-a", str(w)], capture_output=True, text=True)
    host_s = time.perf_counter() - t0
    assert r.returncode == 0, r.stderr
    with G.GrlGpu(0) as ctx:
        ctx.invert(img, w, n_seqs=k)
        got, info = ctx.invert(img, w, n_seqs=k)
    same = got.tobytes() == open(out, "rb").read()
    return {"host_k": k, "host_reverse_bwt_s": round(host_s, 3), "device_k_ms": round(info["device_ms"], 3), "device_k_path": ["walk", "jump"][info["path"]],
            "host_over_device": round(host_s * 1e3 / info["device_ms"], 1), "host_output_equal": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=",".join(WORKLOADS))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--walk-one-string", action="store_true")
    a = ap.parse_args()
    card = gpu_card()
    for name in a.only.split(","):
        make, host_k = WORKLOADS[name]
        arr = make()
        img = np.empty(16 + arr.size * 16, np.uint8)
        nb, n_runs, sb, fb, binfo = G.build_bwt_packed(arr, img, n_threads=16)
        img_p = pinned(nb)   # image and output in pinned memory: the copies inside device_ms run at full PCIe rate
        img_p[:] = img[:nb]
        img = img_p
        out = pinned(arr.size * arr.dtype.itemsize)
        res = {"workload": name, "gpu": card, "n": int(arr.size), "w": arr.dtype.itemsize, "n_strings": int((arr == arr[-1]).sum()), "n_runs": n_runs,
               "image_bytes": nb, "B": max(4096, arr.size // 2048)}
        for label, flags in (("auto", 0), ("walk", G.FLAG_FORCE_WALK), ("jump", G.FLAG_FORCE_JUMP)):
            if label == "walk" and name == "one" and not a.walk_one_string:
                res[label] = "not measured"
                continue
            res[label] = time_path(img, arr, flags, a.reps, out)
        with tempfile.TemporaryDirectory() as tmp:
            res.update(host_vs_device(img, arr, host_k, tmp))
        print(json.dumps(res), flush=True)
        del arr, img, out


if __name__ == "__main__":
    main()
