"""bench.py on the device: --dump-outputs writes what the timed path computed in its last step, whatever the number of steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import grlbwt_b200 as G

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
READS = 20000
LEVEL = ("rule_l", "rule_r", "has_hocc", "pre_sym", "pre_len")


def run_bench(out, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--reads", str(READS), "--steps", str(steps), "--warmup", "1", "--no-e2e",
                        "--no-cpu-baseline", "--bwt-reads", "0", "--dump-outputs", str(out)], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
    return {n: np.load(out / (n + ".npy")) for n in ("rounds", "final_parse") + tuple("last_" + k for k in LEVEL)}


def test_dump_outputs_are_the_parse_phase_of_the_bench_text(tmp_path):
    one, three = run_bench(tmp_path / "one", 1), run_bench(tmp_path / "three", 3)
    for name, a in one.items():
        assert a.dtype == np.float64 and np.array_equal(a, three[name]), name
    import torch
    import bench
    text = bench.make_reads_on_device(torch, 0, READS, 42, torch.device("cuda", 0)).cpu().numpy()
    rows = []
    with G.GrlGpu(0) as ctx:
        ctx.set_text(text)
        while True:
            r = ctx.round()
            rows.append([r.round, r.n_in, r.parse_len, r.n_phrases, r.dict_syms, r.tot_phrases, r.n_pre_runs])
            if r.done:
                break
        level, parse = ctx.fetch_level(), ctx.fetch_parse()
    assert np.array_equal(one["rounds"], np.array(rows, np.float64))
    assert np.array_equal(one["final_parse"], parse.astype(np.float64)) and parse.size == READS
    for k in LEVEL:
        assert np.array_equal(one["last_" + k], level[k].astype(np.float64)), k
