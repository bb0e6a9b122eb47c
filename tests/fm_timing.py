"""Timing of the FM-index on the device (grlgpu_fm_load / _count / _locate), one JSON line per workload.

Each workload is built with build_bwt_packed in the same command. Timed, by CUDA events on the context's stream (device_ms of the
call: pattern upload, search, locate, result download): the load; count of 10^6 length-32 patterns sampled from the strings, of
10^6 random length-32 patterns and of 10^5 length-150 patterns sampled from the strings; locate of 10^5 sampled length-32
patterns. On the reads locate takes the walk; on the long genomes it takes the table, timed as the first call after a load (the
table is built inside it) and as a second call. One warm-up, then the median of `--reps`. The host tool fm_query answers the
first 10^4 patterns of the sampled length-32 set (wall clock of the process, .rl_bwt reading and per-symbol run lists included)
and its output must equal the device's bytes for the same patterns (counts with -l on the reads, counts only on the long genomes,
where each host locate walks millions of LF steps). tests/invert_timing.py is re-run afterwards in the same command, so the
inversion, which shares the LF-table build with the load, is measured on the same card. The GPU name and power limit are read
by nvidia-smi in the same command.

    python tests/fm_timing.py [--out profiles/r04_fm_timing.jsonl] [--only reads,long] [--reps 3] [--invert reads,long]
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


def sample(arr, rng, n_pat, m):
    """n_pat windows of m symbols inside the strings (strings shorter than m are never chosen) -> (cells, offsets)"""
    sep = arr[-1]
    ends = np.flatnonzero(arr == sep)
    starts = np.concatenate(([0], ends[:-1] + 1))
    ok = np.flatnonzero(ends - starts >= m)
    k = rng.choice(ok, n_pat)
    p = starts[k] + (rng.random(n_pat) * (ends[k] - starts[k] - m + 1)).astype(np.int64)
    cells = arr[(p[:, None] + np.arange(m)).ravel()]
    return cells, np.arange(0, n_pat * m + 1, m, dtype=np.uint64)


def median_of(fn, reps, key="device_ms"):
    """one warm-up, then `reps` calls of fn (each returns an info dict) -> (their dicts, median of info[key])"""
    fn()
    runs = [fn() for _ in range(reps)]
    return runs, float(np.median([r[key] for r in runs]))


def host_check(img, arr, cells, off, tmp, locate):
    sep = int(arr[-1])
    rl, pp = os.path.join(tmp, "x.rl_bwt"), os.path.join(tmp, "p.bin")
    img.tofile(rl)
    n = off.size - 1
    with open(pp, "wb") as f:
        f.write(np.insert(cells.reshape(n, -1), cells.size // n, sep, axis=1).astype(arr.dtype).tobytes())
    flags = ["-l"] if locate else []
    t0 = time.perf_counter()
    h = subprocess.run([os.path.join(G.LIB_DIR, "fm_query"), rl, pp] + flags, capture_output=True)
    host_s = time.perf_counter() - t0
    assert h.returncode == 0, h.stderr
    t0 = time.perf_counter()
    d = subprocess.run([os.path.join(G.LIB_DIR, "fm_query_gpu"), rl, pp] + flags, capture_output=True)
    tool_s = time.perf_counter() - t0
    assert d.returncode == 0, d.stderr
    return {"host_n_pat": n, "host_locate": locate, "host_fm_query_s": round(host_s, 3), "fm_query_gpu_s": round(tool_s, 3),
            "host_output_equal": h.stdout == d.stdout}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_fm_timing.jsonl"))
    ap.add_argument("--only", default=",".join(WORKLOADS))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--invert", default="reads,long", help="workloads of tests/invert_timing.py to re-run afterwards ('' for none)")
    a = ap.parse_args()
    card = gpu_card()
    lines = []
    for name in a.only.split(","):
        arr = WORKLOADS[name]()
        img = np.empty(16 + arr.size * 16, np.uint8)
        nb, n_runs, sb, fb, _ = G.build_bwt_packed(arr, img, n_threads=16)
        img = img[:nb].copy()
        rng = np.random.default_rng(1)
        s32 = sample(arr, rng, 1_000_000, 32)
        r32 = (rng.choice(np.frombuffer(b"ACGT", np.uint8), 32_000_000), s32[1])
        s150 = sample(arr, rng, 100_000, 150)
        loc = (s32[0][:100_000 * 32], s32[1][:100_001])
        res = {"workload": name, "gpu": card, "n": int(arr.size), "n_runs": n_runs, "image_bytes": nb, "B": max(4096, arr.size // 2048)}
        with G.GrlGpu(0) as ctx:
            loads, res["load_ms"] = median_of(lambda: ctx.fm_load(img), a.reps, "load_ms")
            res["sigma"], res["n_strings"] = loads[-1]["sigma"], loads[-1]["n_strings"]
            for key, pats in (("count_sampled32", s32), ("count_random32", r32), ("count_sampled150", s150)):
                last = {}

                def one():
                    sp, ep, d = ctx.fm_count(pats)
                    last["occ"] = int((ep - sp).sum())
                    return d
                runs, med = median_of(one, a.reps)
                n_pat = pats[1].size - 1
                res[key] = {"n_pat": n_pat, "device_ms": round(med, 3), "search_ms": round(float(np.median([r["search_ms"] for r in runs])), 3),
                            "patterns_per_s": round(n_pat / med * 1e3), "n_occ": last["occ"]}
            if name == "reads":
                runs, med = median_of(lambda: ctx.fm_locate(loc)[3], a.reps)
                res["locate_sampled32"] = {"path": ["walk", "table"][runs[-1]["path"]], "n_occ": runs[-1]["n_occ"], "device_ms": round(med, 3),
                                           "locate_ms": round(float(np.median([r["locate_ms"] for r in runs])), 3),
                                           "occ_per_s": round(runs[-1]["n_occ"] / med * 1e3)}
            else:   # the table: first call after a load builds it, the second reuses it
                firsts, seconds = [], []
                for _ in range(a.reps + 1):
                    ctx.fm_load(img)
                    firsts.append(ctx.fm_locate(loc)[3])
                    seconds.append(ctx.fm_locate(loc)[3])
                firsts, seconds = firsts[1:], seconds[1:]
                res["locate_sampled32"] = {"path": ["walk", "table"][firsts[-1]["path"]], "n_occ": firsts[-1]["n_occ"], "jump_rounds": firsts[-1]["jump_rounds"],
                                           "first_call_ms": round(float(np.median([r["device_ms"] for r in firsts])), 3),
                                           "second_call_ms": round(float(np.median([r["device_ms"] for r in seconds])), 3),
                                           "second_path": ["walk", "table"][seconds[-1]["path"]]}
            # device time of the host subset, for the baseline
            sub = (s32[0][:N_HOST * 32], s32[1][:N_HOST + 1])
            if name == "reads":
                _, res["device_subset_ms"] = median_of(lambda: ctx.fm_locate(sub)[3], a.reps)
            else:
                _, res["device_subset_ms"] = median_of(lambda: ctx.fm_count(sub)[2], a.reps)
        with tempfile.TemporaryDirectory() as tmp:
            res.update(host_check(img, arr, *sub, tmp, name == "reads"))
        print(json.dumps(res), flush=True)
        lines.append(json.dumps(res))
        del arr, img
    inv = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "invert_timing.py"), "--only", a.invert], capture_output=True, text=True) if a.invert else None
    assert inv is None or inv.returncode == 0, inv.stderr
    for ln in (inv.stdout.splitlines() if inv else []):
        if ln.startswith("{"):
            lines.append(json.dumps({"invert_timing": json.loads(ln)}))
            print(lines[-1], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
