#!/usr/bin/env python
"""bench.py -- parse-phase throughput of the B200 path (BASELINE.json metric: input MB/s to BCR BWT;
parse-round HBM GB/s vs peak) on the C2 workload: synthetic DNA reads, 150 bp, '\\n'-separated.

A "step" = one pass of the hot path over the collection: collection statistics + every parse round
(boundary scan, dedup, dictionary ranking, pre-BWT/grammar, rewrite) until each string is one
metasymbol, i.e. what exact_algo::par_phase does in the reference.
  value : text already resident in HBM (grlgpu_set_text_device), nothing copied.
  e2e   : through the C ABI with HOST buffers: pinned text -> device every step, every level's
          artefacts (rules, hocc marks, preliminary BWT) and the final parse copied back to host.
  --impl reference : the UNMODIFIED reference parse phase (oracle/_ref/ref_harness = its par_phase,
          built from /root/reference by oracle/Makefile) on the host cores, on a bounded sample.
One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "input MB/s through the parse phase of the BCR BWT construction (all grammar rounds on device); whole construction: bwt_total"
READ_LEN = 150


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=50_000_000, help="reads of the collection (C2: 50M x 150 bp = 7.55 GB)")
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c5"],
                    help="c2: random reads (the metric's config); c3: repetitive genomes (BASELINE.json configs[2]); c5: 200M short + 10%% long reads, 33 GB (configs[4], needs 8 GPUs)")
    ap.add_argument("--c5-blocks", type=int, default=302_114, help="c5: blocks of 662 reads x 150 bp + one 10 kbp read (302114 blocks = 200M short reads, 33.2 GB)")
    ap.add_argument("--copies", type=int, default=1000, help="c3: genome copies")
    ap.add_argument("--genome", type=int, default=4_000_000, help="c3: genome length")
    ap.add_argument("--sample-reads", type=int, default=1_000_000, help="reads of the bounded CPU-baseline / same-sample leg (151 MB)")
    ap.add_argument("--ref-budget-s", type=float, default=240.0, help="--impl reference: wall-clock budget of the whole run; the per-step sample is sized to fit")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--bwt-reads", type=int, default=8_000_000, help="reads of the whole-construction leg (bwt_total); 0 skips it")
    ap.add_argument("--write-digest", action="store_true", help="1 GPU: store the output digest under profiles/ as the value every rank count must reproduce")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--comm", choices=["auto", "ipc", "nccl"], default="auto",
                    help="exchange backend of the N > 1 ranks: CUDA IPC windows + shared-memory rendezvous (one box, NVLink), or NCCL send/recv")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64): rounds (per round: round, n_in, "
                         "parse_len, n_phrases, dict_syms, tot_phrases, n_pre_runs), the last level (last_rule_l, last_rule_r, last_has_hocc, "
                         "last_pre_sym, last_pre_len) and final_parse; an array longer than 2^20 values is replaced by the values at the sorted "
                         "positions numpy.random.default_rng(0).integers(0, length, 2^20)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def c2_workload_desc(reads):
    return f"C2: {reads} reads x {READ_LEN} bp uniform ACGT + newline ({reads * (READ_LEN + 1) / 1e9:.3f} GB), BASELINE.json configs[1]"


# ---------------------------------------------------------------- reference / CPU baseline
def cpu_parse_phase(sample_reads, threads, repeats=1):
    """time the reference's own parse phase on `sample_reads` C2-shaped reads; -> (MB/s, kind, sample description)"""
    import numpy as np
    import gen
    arr = gen.dna_reads(sample_reads, READ_LEN, seed=42)
    from oracle import refbin
    harness = refbin.ref_path("ref_harness")
    desc = f"{sample_reads} reads x {READ_LEN} bp ({arr.nbytes / 1e6:.1f} MB), tests/gen.dna_reads seed 42"
    secs = []
    if harness:
        with tempfile.TemporaryDirectory(dir="/tmp") as td:
            inp = os.path.join(td, "sample.txt")
            arr.tofile(inp)
            for _ in range(repeats):
                r = subprocess.run([harness, "parse", inp, "1", str(threads), td], capture_output=True, text=True, cwd=td)
                t = [ln for ln in r.stdout.splitlines() if ln.startswith("PAR_PHASE_SECONDS")]
                if r.returncode != 0 or not t:
                    raise RuntimeError("reference harness failed: " + (r.stdout + r.stderr)[-400:])
                secs.append(float(t[0].split()[1]))
        return [arr.nbytes / 1e6 / s for s in secs], "reference", desc + f"; unmodified reference par_phase, -t {threads}, built {refbin.ref_flags()}", threads
    from oracle import oracle as O  # port (single thread)
    for _ in range(repeats):
        t0 = time.time()
        o = O.Oracle(arr)
        o.par_phase()
        secs.append(time.time() - t0)
        o.close()
    return [arr.nbytes / 1e6 / s for s in secs], "port", desc + "; oracle/oracle.c restatement, 1 thread", 1


def run_reference(args, rank):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    total = args.warmup + args.steps
    # every step is one run of the reference's parse phase on a bounded sample; the sample is as large as the budget of the
    # whole run allows (the reference parses ~5 MB/s on reads and gets slower with size, so larger samples flatter it less)
    per_step_s = max(2.0, args.ref_budget_s / max(1, total) - 1.0)
    args.sample_reads = int(min(args.sample_reads, max(100_000, per_step_s * 4.0e6 / (READ_LEN + 1))))
    rates, kind, desc, cores = cpu_parse_phase(args.sample_reads, threads, repeats=total)
    timed = rates[args.warmup:]
    # the reference's whole program (parse + induction + output) on the same sample, once, for context
    bwt_total = None
    from oracle import refbin
    exe = refbin.ref_path("grlbwt_ref")
    if exe and args.ref_budget_s >= 60:
        import gen
        arr = gen.dna_reads(args.sample_reads, READ_LEN, seed=42)
        with tempfile.TemporaryDirectory(dir="/tmp") as td:
            inp = os.path.join(td, "sample.txt")
            arr.tofile(inp)
            t0 = time.time()
            r = subprocess.run([exe, inp, "-t", str(threads), "-T", td], cwd=td, capture_output=True, text=True)
            dt = time.time() - t0
            if r.returncode == 0:
                bwt_total = {"value": round(arr.nbytes / 1e6 / dt, 3), "unit": "MB/s", "sample": desc, "what": "reference grlbwt CLI, text file -> .rl_bwt file"}
    sample_mb = args.sample_reads * (READ_LEN + 1) / 1e6
    ms = [sample_mb / r * 1e3 for r in timed]
    val = sample_mb * len(timed) / (sum(ms) / 1e3)
    line = {"impl": "reference", "metric": METRIC, "value": round(val, 3), "unit": "MB/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(sum(ms) / len(ms), 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": c2_workload_desc(args.reads), "sample": desc, "same_config": False,
                       "timing": "host wall clock around par_phase inside the harness; each step = one bounded sample of the workload"},
            "cpu_baseline": {"value": round(val, 3), "unit": "MB/s", "cores": cores, "kind": kind, "sample": desc},
            "e2e": {"value": round(val, 3), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
            "bwt_total": bwt_total}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi polling the job's GPUs every 100 ms from ONE process (rank 0). It is started before the warm-up steps, so that its
    start-up (NVML initialisation takes driver-wide locks) stays outside the timed region; only the rows between mark() and stop() count."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, indices):
        self.rows, self.proc, self.indices, self.first = [], None, list(indices), 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", ",".join(str(i) for i in self.indices), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def mark(self):
        self.first = len(self.rows)

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        rows = self.rows[self.first:] or self.rows[-len(self.indices):]   # a region shorter than one polling period: the latest sample
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "gpus": self.indices}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm), "gpus": self.indices}


# ---------------------------------------------------------------- our arm
GEN_BLOCK_READS = 250_000


def make_reads_on_device(torch, first_read, n_reads, seed, device):
    """Reads [first_read, first_read + n_reads) of THE collection defined by `seed` (uniform ACGT + '\\n'; shape of
    tests/gen.dna_reads, torch RNG). The collection is generated in fixed blocks of GEN_BLOCK_READS reads, block b from
    the generator state seed * 1000003 + b, whatever slice is asked for: N ranks build slices of the SAME global text,
    so the output of an N-rank job can be compared with the 1-rank job (digest in the JSON line)."""
    g = torch.Generator(device=device)
    lut = torch.tensor([65, 67, 71, 84], dtype=torch.uint8, device=device)
    out = torch.empty((n_reads, READ_LEN + 1), dtype=torch.uint8, device=device)
    B = GEN_BLOCK_READS
    for b in range(first_read // B, (first_read + n_reads - 1) // B + 1):
        g.manual_seed(seed * 1_000_003 + b)
        idx = torch.randint(0, 4, (B, READ_LEN), generator=g, device=device, dtype=torch.int64)  # always the whole block
        lo, hi = max(first_read, b * B), min(first_read + n_reads, (b + 1) * B)
        out[lo - first_read: hi - first_read, :READ_LEN] = lut[idx[lo - b * B: hi - b * B]]
        del idx
    out[:, READ_LEN] = 10
    return out.reshape(-1)


def make_genomes_on_device(torch, first_copy, n_copies, genome_len, seed, device, snp=1e-3, dele=1e-4):
    """Copies [first_copy, first_copy + n_copies) of the C3 collection: one random genome (seed 7), copy i mutated from the
    generator state seed * 1000003 + i (substitutions + single-base deletions; shape of tests/gen.repetitive_genomes), so
    every rank count sees the same global text"""
    gb = torch.Generator(device=device)
    gb.manual_seed(7)
    base = torch.randint(0, 4, (genome_len,), generator=gb, device=device, dtype=torch.int64)
    g = torch.Generator(device=device)
    lut = torch.tensor([65, 67, 71, 84], dtype=torch.uint8, device=device)
    nl = torch.tensor([10], dtype=torch.uint8, device=device)
    parts = []
    for i in range(first_copy, first_copy + n_copies):
        g.manual_seed(seed * 1_000_003 + i)
        s = base.clone()
        m = torch.rand(genome_len, generator=g, device=device) < snp
        s[m] = (s[m] + torch.randint(1, 4, (int(m.sum()),), generator=g, device=device)) % 4
        keep = torch.rand(genome_len, generator=g, device=device) >= dele
        parts.append(lut[s[keep]])
        parts.append(nl)
    return torch.cat(parts)


C5_SHORT, C5_LONG, C5_CHUNK = 662, 10_000, 512   # a block = 662 short reads + one long read (10 % of the bases); generated 512 blocks at a time
C5_BLOCK_BYTES = C5_SHORT * (READ_LEN + 1) + C5_LONG + 1


def make_mixed_on_device(torch, first_chunk, n_chunks, total_blocks, seed, device):
    """Chunks [first_chunk, first_chunk + n_chunks) of the C5 collection (shape of tests/gen.mixed_reads: short reads with a long
    read interleaved deterministically after every 662 of them); chunk c covers blocks [512 c, 512 (c+1)) and comes from the
    generator state seed * 1000003 + c, so every rank count sees the same global text"""
    g = torch.Generator(device=device)
    lut = torch.tensor([65, 67, 71, 84], dtype=torch.uint8, device=device)
    parts = []
    for c in range(first_chunk, first_chunk + n_chunks):
        nb = min(C5_CHUNK, total_blocks - c * C5_CHUNK)
        g.manual_seed(seed * 1_000_003 + c)
        blk = torch.empty((nb, C5_BLOCK_BYTES), dtype=torch.uint8, device=device)
        short = blk[:, : C5_SHORT * (READ_LEN + 1)].view(nb, C5_SHORT, READ_LEN + 1)
        short[:, :, :READ_LEN] = lut[torch.randint(0, 4, (C5_CHUNK, C5_SHORT, READ_LEN), generator=g, device=device, dtype=torch.int64)[:nb]]
        short[:, :, READ_LEN] = 10
        lng = blk[:, C5_SHORT * (READ_LEN + 1):]
        lng[:, :C5_LONG] = lut[torch.randint(0, 4, (C5_CHUNK, C5_LONG), generator=g, device=device, dtype=torch.int64)[:nb]]
        lng[:, C5_LONG] = 10
        parts.append(blk.reshape(-1))
    return torch.cat(parts)


def split_range(total, world, rank):
    """contiguous ranges of whole strings, as even as possible (the reference's mt split, parsing_strategies.h:208-214)"""
    per, extra = divmod(total, world)
    first = rank * per + min(rank, extra)
    return first, per + (1 if rank < extra else 0)


DUMP_VALUES = 1 << 20   # per array: the seven float64 arrays of --dump-outputs stay under 64 MB


def dump_outputs(out_dir, ctx, rounds, final_cells, rank, world, dist, host_group):
    """--dump-outputs: what the last step left in the context (the level of its last round and the final parse; N ranks: every rank's
    part, in rank order) and the figures of its rounds. float64 holds every value exactly: the bench's texts are DNA, so symbols,
    ranks and counts stay far below 2^53."""
    import numpy as np
    names = ("rule_l", "rule_r", "has_hocc", "pre_sym", "pre_len")
    if world == 1:
        level, parse = ctx.fetch_level(), ctx.fetch_parse()
    else:
        parts = [None] * world if rank == 0 else None
        dist.gather_object((ctx.mg_fetch_slice(), ctx.fetch_parse_local(final_cells)), parts, dst=0, group=host_group)
        if rank != 0:
            return
        level = {k: np.concatenate([p[0][k] for p in parts]) for k in names}
        parse = np.concatenate([p[1] for p in parts])
    keys = ("round", "n_in", "parse_len", "n_phrases", "dict_syms", "tot_phrases", "n_pre_runs")
    arrays = {"rounds": np.array([[r[k] for k in keys] for r in rounds]), "final_parse": parse}
    arrays.update({"last_" + k: level[k] for k in names})
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if a.size > DUMP_VALUES:
            a = a[np.sort(np.random.default_rng(0).integers(0, a.size, DUMP_VALUES))]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def run_ours(args, rank, world, local_rank):
    import hashlib
    import numpy as np
    import torch
    import torch.distributed as dist
    import grlbwt_b200 as G
    from grlbwt_b200 import mg

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the parse phase has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    host_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        host_group = dist.new_group(backend="gloo")   # host-side waits (an NCCL barrier would spin on the GPUs while rank 0 still uses them)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak, peak_src = (peaks["hbm_gbs"], "MEASURED_PEAKS.json (measured copy)") if "hbm_gbs" in peaks else (6650.0, "fallback 6.65 TB/s")

    # strong scaling: ONE global collection (rank-independent generator), split into contiguous ranges of whole strings
    if args.workload == "c2":
        first_read, my_reads = split_range(args.reads, world, rank)
        text = make_reads_on_device(torch, first_read, my_reads, 42, dev)
        n = text.numel()
        n_total = args.reads * (READ_LEN + 1)
        wl_desc = c2_workload_desc(args.reads)
        wl_key = f"c2_{args.reads}"
    elif args.workload == "c5":
        n_chunks_total = (args.c5_blocks + C5_CHUNK - 1) // C5_CHUNK
        first_chunk, my_chunks = split_range(n_chunks_total, world, rank)
        text = make_mixed_on_device(torch, first_chunk, my_chunks, args.c5_blocks, 5, dev)
        n = text.numel()
        n_total = args.c5_blocks * C5_BLOCK_BYTES
        wl_desc = (f"C5: {args.c5_blocks * C5_SHORT} reads x {READ_LEN} bp + {args.c5_blocks} reads x {C5_LONG} bp (10 % of the bases), interleaved "
                   f"({n_total / 1e9:.3f} GB), BASELINE.json configs[4]")
        wl_key = f"c5_{args.c5_blocks}"
    else:
        first_copy, my_copies = split_range(args.copies, world, rank)
        text = make_genomes_on_device(torch, first_copy, my_copies, args.genome, 1000, dev)
        n = text.numel()
        tot = torch.tensor([n], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(tot)
        n_total = int(tot.item())
        wl_desc = f"C3: {args.copies} copies of a {args.genome} bp genome, 0.1% SNPs + 0.01% deletions ({n_total / 1e9:.3f} GB), BASELINE.json configs[2]"
        wl_key = f"c3_{args.copies}x{args.genome}"
    torch.cuda.synchronize()
    stream = torch.cuda.Stream(device=dev)   # the library issues every kernel (and NCCL call) on this stream, so torch events bracket it
    torch.cuda.set_stream(stream)
    ctx = G.GrlGpu(local_rank, 0, stream=stream.cuda_stream)
    comm = mg.comm_from_torch(dist, rank, world, local_rank, torch, kind=args.comm) if world > 1 else None
    arena = [None]
    final_cells = [0]   # cells of this rank's final parse (one per local string)
    e2e_parts = {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_phase(fetch, collect=None, digest=None, slices=None):
        """all rounds on the text set in ctx. fetch: copy this rank's part of every level + its final parse to the host
        (pinned arena, copies overlapped with the next round); digest: per-round checksums + final parse for the N-identity check"""
        d2h, a_off = 0, 0
        if world == 1:
            ctx.stats()
        else:
            ctx.mg_stats(comm)
        while True:
            r = ctx.round() if world == 1 else ctx.mg_round(comm)
            if collect is not None:
                collect.append(r.as_dict())
            narrow = r.n_in + r.parse_len < (1 << 32)  # run lengths of the level fit 32 bits, as the C++ host fetches them
            if world == 1:
                tot_l, pre_l, plen_l = r.tot_phrases, r.n_pre_runs, r.parse_len
            else:
                sl = ctx.mg_slice_info()
                tot_l, pre_l, plen_l = sl.tot_local, sl.n_pre_local, sl.parse_len_local
                if collect is not None:
                    collect[-1]["exchange_bytes_sent"] = sl.exchange_bytes
                if slices is not None:
                    slices.append((tot_l, pre_l))
            if digest is not None:
                cs = ctx.level_checksum() if world == 1 else ctx.mg_slice_checksum()
                if world > 1:
                    t = torch.from_numpy(np.array(cs, np.uint64).view(np.int64)).to(dev)
                    dist.all_reduce(t)   # sums mod 2^64: the slices of a level add up to the single-GPU value
                    cs = [int(x) for x in t.cpu().numpy().view(np.uint64)]
                digest.append([r.tot_phrases, r.n_pre_runs, r.parse_len, r.n_phrases, r.dict_syms] + cs)
            if fetch:
                e2e_parts.setdefault("round_ms", []).append(round(r.device_ms, 1))
                if world == 1:
                    ctx.fetch_level(arena[0], async_=True, offset=a_off, narrow_len=True)
                else:
                    ctx.mg_fetch_slice(arena[0], offset=a_off, narrow_len=narrow, async_=True)
                a_off = ctx.arena_end
                d2h += tot_l * (2 * r.sym_bytes + 1) + pre_l * (r.sym_bytes + (4 if narrow else 8))
            if r.done:
                final_cells[0] = plen_l
                if fetch:
                    t_tail = time.perf_counter()
                    ctx.fetch_wait()
                    d2h += ctx.fetch_parse_local(plen_l, arena[0][a_off:]).nbytes
                    e2e_parts["tail_wait_ms"] = (time.perf_counter() - t_tail) * 1e3
                if digest is not None:
                    part = ctx.fetch_parse_local(plen_l).astype(np.uint64)
                    if world > 1:
                        parts = [None] * world if rank == 0 else None
                        dist.gather_object(part, parts, dst=0, group=host_group)
                        part = np.concatenate(parts) if rank == 0 else None
                    digest.append(hashlib.sha256(part.tobytes()).hexdigest() if part is not None else None)
                return d2h

    def step_resident(collect=None, digest=None, slices=None):
        ctx.set_text_device(text.data_ptr(), n, 1)
        run_phase(False, collect, digest, slices)

    # ---- value: text resident in HBM ----
    sampler = ClockSampler(range(world)) if rank == 0 else None   # one nvidia-smi for all the job's GPUs, started ahead of the timed region
    if sampler is not None:
        sampler.start()
    for _ in range(args.warmup):
        step_resident()
    rounds_info, digest, slice_sizes = [], [], []
    step_resident(rounds_info, digest, slice_sizes)   # untimed: per-round figures, output digest
    ctx.profile_reset(); ctx.profile_enable(True)
    step_resident()                      # untimed: per-kernel CUDA-event timing enabled
    prof = ctx.profile()
    ctx.profile_enable(False); ctx.profile_reset()

    barrier()
    if sampler is not None:
        sampler.mark()
    ci0 = comm.info() if comm is not None else None
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    last_rounds = []
    e0.record(stream)
    for i in range(args.steps):
        step_resident(last_rounds if args.dump_outputs and i == args.steps - 1 else None)
    e1.record(stream)
    barrier()
    launches = ctx.launch_count() - l0
    exchange_per_step = None
    if comm is not None:
        ci1 = comm.info()
        exchange_per_step = {"rank": rank, "GB_sent": round((ci1["bytes_sent"] - ci0["bytes_sent"]) / args.steps / 1e9, 3),
                             "ms_in_bulk_exchanges": round((ci1["ms_in_bulk"] - ci0["ms_in_bulk"]) / args.steps, 1),
                             "ms_in_small_gathers": round((ci1["ms_in_small"] - ci0["ms_in_small"]) / args.steps, 1),
                             "bulk_exchanges": (ci1["bulk_collectives"] - ci0["bulk_collectives"]) // args.steps,
                             "small_gathers": (ci1["small_collectives"] - ci0["small_collectives"]) // args.steps, "backend": ci1["kind"],
                             "note": "host wall time of rank 0 inside the exchanges, from 'my data is ready' to 'all of it has arrived' (includes waiting for peers)"}
    clocks = sampler.stop() if sampler is not None else None
    ms_total = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    value = n_total * args.steps / 1e6 / (ms_total / 1e3)
    if args.dump_outputs:   # before the e2e steps reuse the context
        dump_outputs(args.dump_outputs, ctx, last_rounds, final_cells[0], rank, world, dist, host_group)

    # ---- e2e: host buffers through the C ABI (pinned text -> device; this rank's levels + final parse -> pinned host) ----
    e2e = None
    if not args.no_e2e:
        host_text = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        host_text.copy_(text)
        torch.cuda.synchronize()
        host_np = host_text.numpy()
        if world == 1:
            need = sum(r["tot_phrases"] * 9 + r["n_pre_runs"] * 12 + 256 for r in rounds_info)
        else:
            need = sum(int(t_ * 9 * 1.05) + int(p_ * 12 * 1.05) + 4096 for t_, p_ in slice_sizes)
        need += (final_cells[0] + 1024) * 8 + (1 << 20)
        arena[0] = torch.empty(int(need), dtype=torch.uint8, pin_memory=True).numpy()
        d2h_bytes = [0]

        def step_e2e():
            e2e_parts.clear()
            t_a = time.perf_counter()
            ctx.set_text(host_np)
            t_b = time.perf_counter()
            d2h_bytes[0] = run_phase(True)
            e2e_parts["h2d_ms"] = (t_b - t_a) * 1e3
            e2e_parts["rounds_and_fetch_ms"] = (time.perf_counter() - t_b) * 1e3

        step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        if world > 1:
            t = torch.tensor([wall_ms, float(n), float(d2h_bytes[0])], device=dev, dtype=torch.float64)
            tm = t.clone()
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            wall_ms, h2d_b, d2h_b = float(tm[0]), int(t[1]), int(t[2])
        else:
            h2d_b, d2h_b = n, d2h_bytes[0]
        e2e = {"value": round(n_total * args.steps / 1e6 / (wall_ms / 1e3), 3), "unit": "MB/s", "h2d_bytes_per_step": int(h2d_b),
               "d2h_bytes_per_step": int(d2h_b), "ms_per_step": round(wall_ms / args.steps, 3),
               "what": "every rank copies its shard from pinned host memory to its GPU and copies its part of every level (rules, hocc marks, "
                       "preliminary BWT) and of the final parse back to pinned host memory; bytes are summed over the ranks",
               "timing": "host wall clock between stream synchronisations, max over ranks",
               "last_step_parts_ms": {k: (list(v) if isinstance(v, list) else round(v, 1)) for k, v in e2e_parts.items()}}
        del host_text

    # ---- same sample as the reference arm / cpu_baseline (numpy generator, host buffers), 1 GPU only ----
    same_sample = None
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            import gen
            sample = gen.dna_reads(args.sample_reads, READ_LEN, seed=42)
            pin = torch.from_numpy(sample).pin_memory().numpy()
            need = 40 * sample.nbytes // 10 + (1 << 22)
            arena[0] = torch.empty(int(need), dtype=torch.uint8, pin_memory=True).numpy()
            ts = []
            for _ in range(4):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ctx.set_text(pin)
                run_phase(True)
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t0)
            ours = sample.nbytes / 1e6 / min(ts[1:])
            rates, kind, desc, cores = cpu_parse_phase(args.sample_reads, os.cpu_count() or 1, repeats=1)
            cpu = {"value": round(rates[0], 3), "unit": "MB/s", "cores": cores, "kind": kind, "sample": desc}
            same_sample = {"sample": f"{args.sample_reads} reads x {READ_LEN} bp ({sample.nbytes / 1e6:.1f} MB), tests/gen.dna_reads seed 42: the identical bytes for both",
                           "ours_e2e_MBps": round(ours, 1), "reference_MBps": round(rates[0], 3), "ratio": round(ours / rates[0], 1),
                           "what": "parse phase, host buffers in / levels out (ours, best of 3 after one warm-up) vs the reference's par_phase with -t = all host cores"}
        except Exception as e:  # the baseline is reporting only
            cpu = {"value": None, "unit": "MB/s", "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {e}"}
    info_comm = comm.info() if comm is not None else None
    if comm is not None:
        comm.close()
    ctx.close()
    arena[0] = None
    del text
    torch.cuda.empty_cache()

    # ---- roofline of the dominant kernel (CUDA events on the launch stream, live, one profiled step) ----
    roof = None
    if prof:
        name, (nl, ms, by) = max(prof.items(), key=lambda kv: kv[1][1])
        achieved = by / 1e9 / (ms / 1e3) if ms > 0 else 0.0
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
        if os.path.exists(tpath) and args.workload == "c2" and args.reads == 50_000_000 and world == 1:
            tj = json.load(open(tpath))
            if tj.get("kernel") == name:   # ncu DRAM bytes of the same kernel on the same workload, per launch
                traffic, traffic_src = round(tj["traffic_bytes_per_launch"]), "profiles/r02_ncu_traffic.json (ncu dram__bytes_read+write, mean over the step's launches)"
        roof = {"bound": "hbm", "kernel": name, "launches_per_step": nl, "avg_launch_ms": round(ms / max(nl, 1), 4), "achieved": round(achieved, 1),
                "peak": hbm_peak, "unit": "GB/s", "frac": round(achieved / hbm_peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                "bytes_per_launch": round(by / max(nl, 1)), "peak_source": peak_src,
                "share_of_step": round(ms / sum(v[1] for v in prof.values()), 4),
                "bytes_model": "expected DRAM bytes of the kernel's launches (SURVEY.md 8d traffic table; DESIGN.md kernels section)"}
    alg_bytes = sum(r["algorithmic_bytes"] for r in rounds_info)
    round_ms = sum(r["device_ms"] for r in rounds_info)
    if world > 1:   # B_r is a per-rank share in multi-GPU rounds: aggregate GB/s = sum over ranks / max time
        t = torch.tensor([float(alg_bytes)], device=dev, dtype=torch.float64)
        dist.all_reduce(t)
        alg_bytes = float(t.item())
        t = torch.tensor([round_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        round_ms = float(t.item())
    keys = ("round", "n_in", "parse_len", "n_phrases", "dict_syms", "tot_phrases", "n_pre_runs", "device_ms", "text_pass_ms", "dict_ms", "rewrite_ms",
            "algorithmic_bytes", "exchange_bytes_sent")
    parse_rounds = {"algorithmic_GB": round(alg_bytes / 1e9, 3), "device_ms": round(round_ms, 3),
                    "achieved_GBps": round(alg_bytes / 1e6 / round_ms, 1) if round_ms else None,
                    "frac_of_measured_peak": round(alg_bytes / 1e6 / round_ms / (hbm_peak * world), 4) if round_ms else None,
                    "frac_of_nominal_8TBps": round(alg_bytes / 1e6 / round_ms / (8000.0 * world), 4) if round_ms else None,
                    "scope": "bytes summed over the ranks, time = max over ranks; per_round lists rank 0's share" if world > 1 else "whole job",
                    "per_round": [{k: (round(v, 3) if isinstance(v, float) else v) for k, v in r.items() if k in keys} for r in rounds_info]}
    kernels = {k: {"launches": v[0], "ms": round(v[1], 3), "model_GBps": round(v[2] / 1e6 / v[1], 1) if v[1] > 0 else None}
               for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])[:14]}
    kernels["(all kernels)"] = {"launches": int(sum(v[0] for v in prof.values())), "ms": round(sum(v[1] for v in prof.values()), 3), "model_GBps": None}

    # ---- output digest: equal for every number of ranks (per-round level checksums + sha256 of the final parse) ----
    dg = None
    if rank == 0:
        h = hashlib.sha256(json.dumps(digest).encode()).hexdigest()
        dpath = os.path.join(ROOT, "profiles", f"digest_{wl_key}.json")
        expected = None
        if os.path.exists(dpath):
            expected = json.load(open(dpath)).get("sha256")
        elif world == 1 and args.write_digest:
            json.dump({"workload": wl_desc, "n_gpus": 1, "sha256": h, "per_round": digest[:-1], "final_parse_sha256": digest[-1]}, open(dpath, "w"), indent=1)
        n_ins = [n_total] + [d_[2] for d_ in digest[:-2]]
        covers = all(d_[7] == n_in_ for d_, n_in_ in zip(digest[:-1], n_ins))
        dg = {"sha256": h, "rounds": len(digest) - 1, "pre_bwt_covers_every_level": covers, "final_parse_sha256": digest[-1], "per_round_tot_phrases": [d[0] for d in digest[:-1]],
              "expected_from_1_gpu": expected, "matches_1_gpu": (h == expected) if expected else None,
              "invariant": "pre_bwt_covers_every_level: the run lengths of level r's preliminary BWT sum to the number of cells of round r's text (checked on the "
                           "checksums, at full size, for every rank count)",
              "what": "sha256 over [tot_phrases, pre-BWT runs, parse length, distinct phrases, dictionary symbols, 4 checksums of rules/hocc/pre-BWT] of every "
                      "round + sha256 of the final parse in string order; the N-rank job parses slices of the same global text, so the value is the same for "
                      "1, 2, 4 and 8 GPUs (profiles/digest_*.json holds the 1-GPU value)"}

    # ---- whole construction: device parse phase + multi-threaded host induction (C++ host, host text -> run-length BCR BWT) ----
    bwt_total = None
    if world > 1:
        dist.barrier(group=host_group)   # every rank has released its device memory
    if rank == 0 and not args.no_e2e and args.workload == "c2" and args.bwt_reads > 0:
        try:
            import gen
            thr = os.cpu_count() or 1
            sample = torch.from_numpy(gen.dna_reads(min(args.reads, args.bwt_reads), READ_LEN, seed=42)).pin_memory().numpy()
            devs = list(range(world))
            # caller-owned pinned landing zone for the image of the .rl_bwt file, reused from call to call: 16-byte header + one record per
            # run (a run per symbol at most) of 1 symbol byte + as many length bytes as the largest symbol frequency needs
            image = torch.empty(16 + (1 + (int(sample.size).bit_length() + 7) // 8) * sample.size, dtype=torch.uint8, pin_memory=True).numpy()
            G.build_bwt_packed(sample[: 151 * 1000], image, devices=devs, n_threads=thr)  # warm the libraries
            best = None
            for _ in range(2):
                t0 = time.perf_counter()
                nb, n_runs, sb, fb, info = G.build_bwt_packed(sample, image, devices=devs, n_threads=thr)
                wall = (time.perf_counter() - t0) * 1e3
                if best is None or wall < best[0]:
                    best = (wall, n_runs, info, nb, sb, fb)
            wall, n_runs, info, nb, sb, fb = best
            hdr = image[:16].view(np.uint64)
            assert nb == 16 + n_runs * (sb + fb) and int(hdr[0]) == sb and int(hdr[1]) == fb
            bwt_total = {"value": round(sample.nbytes / 1e6 / (wall / 1e3), 3), "unit": "MB/s", "n_gpus": world,
                         "sample": f"{sample.size // 151} reads x {READ_LEN} bp ({sample.nbytes / 1e6:.0f} MB)", "wall_ms": round(wall, 1),
                         "h2d_ms": round(info["h2d_ms"], 1), "parse_phase_ms": round(info["par_phase_ms"], 1), "induction_ms": round(info["ind_phase_ms"], 1),
                         "induction": "device (grlgpu_induce: levels never leave the GPU)" if info.get("induced_on_device") else "host threads",
                         "host_threads": thr, "bwt_runs": int(n_runs), "rl_bwt_bytes": int(nb), "rl_bwt_header": [int(sb), int(fb)],
                         "what": "input MB/s to BCR BWT: pinned host text -> image of the reference's .rl_bwt output file in pinned host memory through the C++ "
                                 "host (grlbwt_build_packed: one host thread per GPU, new device contexts every call -- they adopt the device memory "
                                 "the previous contexts of the process left mapped), wall clock of the call, best of 2; file I/O excluded"}
        except Exception as e:
            bwt_total = {"value": None, "error": str(e)[:300]}

    if rank == 0:
        line = {"metric": METRIC, "value": round(value, 3), "unit": "MB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": round(ms_total / args.steps, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
                "data": "synthetic",
                "config": {"workload": wl_desc,
                           "reads": args.reads if args.workload == "c2" else None, "cache": "the text of every round-1 pass (7.55 GB at the default size) exceeds the 126 MB L2",
                           "generator": "torch CUDA RNG in fixed blocks of reads seeded per block: every rank count parses slices of the same global text",
                           "parallelism": "1 GPU" if world == 1 else
                           f"{world} ranks, contiguous ranges of whole reads; the round's dictionary is PARTITIONED, never replicated: phrases by owner (content hash), "
                           f"suffix entries by first-key range, rules by rank range; all exchanges are issued by libgrlgpu.so "
                           f"({exchange_per_step['backend'] if exchange_per_step else ''}; --comm nccl selects NCCL grouped send/recv)",
                           "exchange_per_step": exchange_per_step},
                "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "same_sample": same_sample,
                "digest": dg, "bwt_total": bwt_total, "parse_rounds": parse_rounds, "kernels": kernels}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier(group=host_group)
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
