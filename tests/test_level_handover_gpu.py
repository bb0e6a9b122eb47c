"""GPU suite (-m gpu) for the level hand-over: every way a round's level leaves a context (fetched synchronously or on the copy
stream, with 64- or 32-bit run lengths, parked for host threads, kept on the device and fetched back) hands over the same arrays,
and grlgpu_level_checksum is the documented sum over them. The multi-GPU part checks that the slices of grlgpu_mg_fetch_slice,
placed at rank_base / pre_first, assemble into the single-GPU level."""
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import grlbwt_b200 as G

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_STATE, ERR_LIMIT = -5, -6
NAMES = ("rule_l", "rule_r", "has_hocc", "pre_sym", "pre_len")


class LevelPtrs(C.Structure):  # grlgpu_level_ptrs_t
    _fields_ = [(k, C.c_void_p) for k in NAMES] + [("tot", C.c_uint64), ("n_pre", C.c_uint64), ("sym_bytes", C.c_uint32), ("len_bytes", C.c_uint32),
                                                    ("device", C.c_int)]


def lib():
    L = G.lib_gpu()
    vp, u64 = C.c_void_p, C.c_uint64
    L.grlgpu_keep_level.argtypes = [vp]
    L.grlgpu_kept_levels.argtypes = [vp]
    L.grlgpu_fetch_kept_level.argtypes = [vp, C.c_int, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64), vp, vp, vp, vp, vp]
    return L


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def checksum(lv, rank_base=0):
    """level_checksum_kernel in numpy: sums mod 2^64"""
    k1, k2 = np.uint64(0x9E3779B97F4A7C15), np.uint64(0xC2B2AE3D27D4EB4F)
    u = np.arange(1, lv["rule_l"].size + 1, dtype=np.uint64) + np.uint64(rank_base)
    rl, rr, hh = (lv[k].astype(np.uint64) for k in ("rule_l", "rule_r", "has_hocc"))
    ps, pl = lv["pre_sym"].astype(np.uint64), lv["pre_len"].astype(np.uint64)
    return [int(np.sum(u * ((rl * k1) ^ (rr * k2)), dtype=np.uint64)), int(np.sum(u * hh, dtype=np.uint64)), int(np.sum(pl, dtype=np.uint64)),
            int(np.sum((ps * k1 + np.uint64(1)) * pl, dtype=np.uint64))]


def as_u64(lv):
    return {k: np.asarray(lv[k]).astype(np.uint64) for k in NAMES}


def pinned(nbytes):
    import torch
    return torch.empty(max(nbytes, 16), dtype=torch.uint8, pin_memory=True).numpy()


def expect_state(ctx):
    with pytest.raises(G.GrlGpuError) as e:
        ctx.fetch_level(widen=False)
    assert e.value.status == ERR_STATE


def level_bytes(r):
    return 3 * r.tot_phrases * 8 + r.tot_phrases + r.n_pre_runs * 16 + 96


def run_method(arr, method):
    """every round of `arr` on a fresh context; the level of each round handed over by `method` -> [(round, level)]"""
    L = lib()
    out = []
    with G.GrlGpu(0) as ctx:
        ctx.set_text(arr)
        while True:
            r = ctx.round()
            lv = None
            if method == "sync":
                lv = ctx.fetch_level(widen=False)
                again = ctx.fetch_level(widen=False)  # a synchronous fetch leaves the level in place
                assert all(np.array_equal(lv[k], again[k]) for k in NAMES)
                assert ctx.level_checksum() == checksum(lv), f"round {r.round}"
            elif method in ("async", "async32"):
                arena = pinned(level_bytes(r) + 64)
                got = ctx.fetch_level(arena, widen=False, async_=True, offset=16, narrow_len=method == "async32")
                assert ctx.arena_end <= arena.size and ctx.arena_end % 16 == 0
                expect_state(ctx)
                ctx.fetch_wait()
                lv = {k: np.array(v) for k, v in got.items()}
                if method == "async32":
                    assert lv["pre_len"].dtype == np.uint32
            elif method == "sync32":
                lv = ctx.fetch_level(widen=False, narrow_len=True)
                assert lv["pre_len"].dtype == np.uint32
                assert ctx.level_checksum() == checksum(lv)
            elif method in ("park8", "park4"):
                lp = LevelPtrs()
                assert L.grlgpu_level_park(ctx._h, 8 if method == "park8" else 4, C.byref(lp)) == 0
                assert (lp.tot, lp.n_pre, lp.sym_bytes, lp.len_bytes, lp.device) == (r.tot_phrases, r.n_pre_runs, r.sym_bytes, 8 if method == "park8" else 4, 0)
                sd, ld = G.api.CELL[lp.sym_bytes], G.api.CELL[lp.len_bytes]
                lv = {"rule_l": np.zeros(lp.tot, sd), "rule_r": np.zeros(lp.tot, sd), "has_hocc": np.zeros(lp.tot, np.uint8), "pre_sym": np.zeros(lp.n_pre, sd),
                      "pre_len": np.zeros(lp.n_pre, ld)}
                for k in NAMES:
                    assert L.grlgpu_copy_to_host(lp.device, ptr(lv[k]), getattr(lp, k), lv[k].nbytes) == 0, k
                expect_state(ctx)
                ctx.fetch_wait()
            elif method == "keep":
                rc = L.grlgpu_keep_level(ctx._h)
                if r.sym_bytes == 8:
                    assert rc == ERR_LIMIT  # the device induction takes 32-bit levels only; the level stays
                    ctx.fetch_level(widen=False)
                else:
                    assert rc == 0
                    expect_state(ctx)
                    out.append((r.round, None))
            else:
                raise AssertionError(method)
            if lv is not None:
                out.append((r.round, lv))
            if r.done:
                break
        if method == "keep":  # the kept levels, in round order
            assert L.grlgpu_kept_levels(ctx._h) == len(out)
            for i, (rnd, _) in enumerate(out):
                A, tot, n_pre = C.c_uint64(), C.c_uint64(), C.c_uint64()
                assert L.grlgpu_fetch_kept_level(ctx._h, i, C.byref(A), C.byref(tot), C.byref(n_pre), None, None, None, None, None) == 0
                lv = {"rule_l": np.zeros(tot.value, np.uint32), "rule_r": np.zeros(tot.value, np.uint32), "has_hocc": np.zeros(tot.value, np.uint8),
                      "pre_sym": np.zeros(n_pre.value, np.uint32), "pre_len": np.zeros(n_pre.value, np.uint64)}
                assert L.grlgpu_fetch_kept_level(ctx._h, i, None, None, None, *(ptr(lv[k]) for k in NAMES)) == 0
                out[i] = (rnd, lv)
    return out


@pytest.mark.parametrize("name", ["mutated_200x5k", "u16_rand", "reads_2000x150", "u64_rand"])
def test_level_handover_paths_agree(all_cases, name):
    ref = dict(run_method(all_cases[name], "sync"))
    assert len(ref) >= 2
    for method in ("async", "sync32", "async32", "park8", "park4", "keep"):
        got = run_method(all_cases[name], method)
        if method != "keep":
            assert [rnd for rnd, _ in got] == sorted(ref), method
        assert got, method
        for rnd, lv in got:
            want = ref[rnd]
            for k in NAMES:
                assert lv[k].dtype.itemsize == want[k].dtype.itemsize or k == "pre_len", (method, rnd, k)
                assert np.array_equal(lv[k].astype(np.uint64), want[k].astype(np.uint64)), (name, method, rnd, k)


MG_WORKER = r'''
import json, os, sys
import numpy as np
import torch
import torch.distributed as dist
ROOT = os.environ["GRL_ROOT"]
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import gen
import grlbwt_b200 as G
from grlbwt_b200 import mg
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(0)
dist.init_process_group("gloo")
comm = mg.comm_from_torch(dist, rank, world, 0, torch, kind="ipc")
arr = gen.small_cases()[os.environ["GRL_CASE"]]
lo, hi = mg.shard_bounds(arr, world)[rank]
ctx = G.GrlGpu(0)
ctx.set_text(arr[lo:hi])
ctx.mg_stats(comm)
rounds = []
while True:
    r = ctx.mg_round(comm)
    cs = ctx.mg_slice_checksum()
    k = len(rounds)
    if k % 2 == 0:   # 64-bit lengths, synchronous: the slice stays and can be fetched again
        sl = ctx.mg_fetch_slice()
        again = ctx.mg_fetch_slice()
        assert all(np.array_equal(sl[n], again[n]) for n in ("rule_l", "rule_r", "has_hocc", "pre_sym", "pre_len"))
        assert ctx.mg_slice_checksum() == cs
    else:            # 32-bit lengths on the copy stream, into pinned memory: the slice is parked until fetch_wait
        arena = torch.empty(1 << 24, dtype=torch.uint8, pin_memory=True).numpy()
        sl = ctx.mg_fetch_slice(arena, offset=16, narrow_len=True, async_=True)
        for call in (ctx.mg_fetch_slice, ctx.mg_slice_checksum):
            try:
                call()
                raise AssertionError("a parked slice was handed over twice")
            except G.GrlGpuError as e:
                assert e.status == -5, e
        ctx.fetch_wait()
        sl = {n: (np.array(v) if isinstance(v, np.ndarray) else v) for n, v in sl.items()}
        assert sl["pre_len"].dtype == np.uint32
    mine = {n: sl[n].astype(np.uint64).tolist() for n in ("rule_l", "rule_r", "has_hocc", "pre_sym", "pre_len")}
    mine.update(rank_base=int(sl["rank_base"]), pre_first=int(sl["pre_first"]), cs=cs)
    parts = [None] * world
    dist.all_gather_object(parts, mine)
    if rank == 0:
        lv = {n: np.zeros(r.tot_phrases if n in ("rule_l", "rule_r", "has_hocc") else r.n_pre_runs, np.uint64) for n in mine if n not in ("rank_base", "pre_first", "cs")}
        filled = {n: np.zeros(a.size, bool) for n, a in lv.items()}
        for p in parts:
            for n in lv:
                at = p["rank_base"] if n in ("rule_l", "rule_r", "has_hocc") else p["pre_first"]
                m = len(p[n])
                assert not filled[n][at:at + m].any(), ("slices overlap", n)
                lv[n][at:at + m] = p[n]
                filled[n][at:at + m] = True
        assert all(f.all() for f in filled.values()), "the slices do not cover the level"
        cs_sum = [sum(p["cs"][i] for p in parts) % (1 << 64) for i in range(4)]
        rounds.append({"level": {n: a.tolist() for n, a in lv.items()}, "cs": cs_sum})
    else:
        rounds.append(None)
    if r.done:
        break
if rank == 0:
    with open(os.environ["GRL_OUT"], "w") as f:
        json.dump(rounds, f)
comm.close(); ctx.close()
dist.destroy_process_group()
'''


def test_mg_fetch_slice_assembles_level(tmp_path, all_cases):
    """three processes share GPU 0 (gloo + CUDA IPC exchange); each round's slices, fetched alternately with 64-bit lengths
    synchronously and 32-bit lengths on the copy stream, assemble into the single-GPU level, and their checksums add up to it"""
    name = "mutated_200x5k"
    ref = []
    with G.GrlGpu(0) as ctx:
        ctx.set_text(all_cases[name])
        while True:
            r = ctx.round()
            ref.append((as_u64(ctx.fetch_level(widen=False)), ctx.level_checksum()))
            if r.done:
                break
    script, out = tmp_path / "w.py", tmp_path / "rounds.json"
    script.write_text(MG_WORKER)
    env = dict(os.environ, GRL_ROOT=ROOT, GRL_CASE=name, GRL_OUT=str(out), GRLGPU_IPC_TIMEOUT_S="120")
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "3", "--master-addr", "127.0.0.1", "--master-port", "29753",
                        str(script)], capture_output=True, text=True, env=env, timeout=600)
    assert p.returncode == 0, (p.stdout + p.stderr)[-3000:]
    got = json.loads(out.read_text())
    assert len(got) == len(ref)
    for rnd, (g, (want, cs)) in enumerate(zip(got, ref), 1):
        for k in NAMES:
            a = np.array(g["level"][k], np.uint64)
            assert np.array_equal(a, want[k]), (rnd, k, hashlib.sha256(a.tobytes()).hexdigest()[:12])
        assert g["cs"] == cs, rnd
        assert cs == checksum(want)
