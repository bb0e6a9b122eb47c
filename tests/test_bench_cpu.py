"""bench.py on a CPU-only box: the reference arm runs (it is the reference's own CPU code), our arm refuses to."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--sample-reads", "3000"],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-500:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "MB/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["steps"] == 1 and line["warmup"] == 1 and line["n_gpus"] == 1 and line["gpu_launches"] == 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] == line["e2e"]["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["metric"].startswith("input MB/s through the parse phase of the BCR BWT construction")
    assert line["config"]["workload"].startswith("C2: 50000000 reads") and "reads x 150 bp" in line["config"]["sample"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--sample-reads", "3000"],
                       capture_output=True, text=True, cwd=ROOT, env=env, timeout=600)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_bad_arguments_are_rejected():
    for bad in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + bad, capture_output=True, text=True, cwd=ROOT, timeout=600)
        assert r.returncode == 2 and bad[0] in r.stderr, (bad, r.stderr[-300:])


def test_our_arm_refuses_to_run_without_a_device():
    import torch
    if torch.cuda.is_available():
        return  # on a GPU box the real bench covers it
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--reads", "1000", "--no-e2e", "--no-cpu-baseline"],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode != 0 and "no CPU fallback" in r.stderr
