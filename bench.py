#!/usr/bin/env python
"""bench.py -- generations/sec of the Pansim Wright-Fisher step (and distances/sec
of the pairwise pass) on B200, with the kernel roofline and the CPU baseline.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm (oracle port)

Workload (BASELINE.json configs[1], "cfg2"): pop_size 1000 x core 1.2 Mbp,
6000 pan genes (4000 accessory), selection on (prop_positive 0.1), competition
0.5, 100 000 sampled pairs. A step = one generation, main.rs:435-464. The
per-generation distance pass of --print_dist (main.rs:502-504) is timed
separately and reported under "distances".

N > 1 (torchrun, one rank per GPU): weak scaling over columns -- every rank holds
all individuals for its own 1.2 Mbp slice of an N x 1.2 Mbp alignment (accessory
matrix replicated), so the job processes N cfg2-shaped slabs per step and `value`
counts slab-generations per second. The generation step needs no collective; the
distance pass sums the per-pair partial core counts with NCCL inside the library
(pansim_comm_init_rank; torch.distributed only carries the 128-byte unique id).

--steps K is the number of generations timed: one device-resident batch of K generations after the
warm-up (at the default K = 100 a window of about 15 ms on a B200 with a 1000 W power limit). --repeats R times R such batches
(R x K generations) and reports the median batch; at the default R = 1 the `repeats` record holds that
one batch. The end-to-end record (`e2e`) is the median of 5 runs whatever R is.

--impl reference runs K full cfg2 generations on the host, a few seconds each: pass a small --steps
for a quick sample.

--dump-outputs DIR writes, after the timed batches, the state a caller of the timed path holds after its
last generation as DIR/<name>.npy (float32 / float64, see dump_outputs). The inputs are seeded, so two
builds run with the same arguments can be compared file by file.

Also in the line:
  repeats        R, and the fastest / median / slowest of the R batches
  shard_parity   (N > 1) a small column-sharded run equals the unsharded one bit for bit; the run
                 fails when it does not
  cfg2_print_dist  the cfg2 step WITH its per-generation distance pass and on-device statistics
  cfg4_strong    BASELINE configs[3] (10 000 x 5 Mbp x 18 000) column-sharded over the N ranks
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

_JSON_OUT = sys.stdout
CFG2 = dict(pop_size=1000, core_size=1_200_000, pan_genes=6000, core_genes=2000, n_gen=100,
            max_distances=100_000, prop_positive=0.1, competition_strength=0.5, seed=0)
PEAK_FALLBACK_GBS = 6650.0      # /opt/skills/guides/B200_PROFILING.md fallback


def ncu_traffic(kernel: str):
    """DRAM bytes per launch of a kernel from the committed ncu capture (profiles/r02_dram_traffic.json,
    made from the CSV files beside it); None when the file or the kernel is missing."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_dram_traffic.json")) as f:
            e = json.load(f)[kernel]
        return e
    except Exception:
        return None


def selection_coefficients(rng, n, prop_positive, pos_lambda=10.0, neg_lambda=10.0):
    """main.rs:289-319 (host side keeps this; numpy generator instead of StdRng)."""
    s = np.zeros(n)
    if prop_positive < 0:
        return s
    for i in range(n):
        if rng.random() <= prop_positive:
            s[i] = rng.exponential(1.0 / pos_lambda)
        else:
            v = rng.exponential(1.0 / neg_lambda)
            while v > 1.0:
                v = rng.exponential(1.0 / neg_lambda)
            s[i] = -v
    return s


def sample_pairs(rng, n, p):
    """main.rs:413-427"""
    r1 = rng.integers(0, n, p).astype(np.uint32)
    r2 = rng.integers(0, n - 1, p).astype(np.uint32)
    r2 = (r2 + (r2 >= r1)).astype(np.uint32)
    return r1, r2


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return PEAK_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi sampler (100 ms). stop(t0, t1) keeps the samples taken while the GPU was under
    load, i.e. between the wall-clock times t0 (start of warm-up) and t1 (end of the e2e loop)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self, t0=None, t1=None):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(parts[1]), float(parts[2]),
                             [n for n, v in zip(names, parts[4:8]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        os.unlink(self.f.name)
        load = [r for r in rows if t0 is not None and t0 - 0.15 <= r[0] <= t1 + 0.15]
        use = load or rows
        if use:
            out = {"sm_mhz": float(np.median([r[1] for r in use])), "sm_max_mhz": float(max(r[2] for r in use)),
                   "reasons": sorted({n for r in use for n in r[3]}), "samples": len(use),
                   "window": "warm-up .. end of e2e loop" if load else "whole run (no sample fell in the load window)"}
        return out


def cpu_baseline_sample(n_gen: int, with_distances: bool, pairs: int):
    """Times the oracle port (CPU restatement of the reference, threads where the
    reference uses rayon) on a bounded sample of the same workload."""
    from oracle import binding as ob
    # all host threads this process may use (torchrun exports OMP_NUM_THREADS=1, so ask the OS)
    try:
        threads = len(os.sched_getaffinity(0))
    except AttributeError:
        threads = os.cpu_count() or 1
    kw = dict(CFG2)
    kw["max_distances"] = pairs
    p = ob.default_params(threads=threads, **kw)
    t_gen, t_dist = ob.time_generations(p, n_gen, with_distances, use_tables=True)
    return threads, t_gen, t_dist


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path. The Rust
    crate cannot be built here (no cargo), so this is the oracle port."""
    if rank != 0:
        return
    # each step = one cfg2 generation on the host cores (a few s each)
    steps_run = args.steps
    pairs = 2000
    threads, t_gen, t_dist = cpu_baseline_sample(args.warmup if args.warmup < 1 else 1, False, pairs)  # warm page cache / omp
    threads, t_gen, t_dist = cpu_baseline_sample(steps_run, True, pairs)
    ms = 1e3 * t_gen / steps_run
    val = steps_run / t_gen
    pairs_per_s = steps_run * pairs / t_dist if t_dist > 0 else None
    line = {
        "impl": "reference", "metric": "generations/sec", "value": val, "unit": "generations/s",
        "n_gpus": args.gpus, "steps": steps_run, "warmup": 1, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "cfg2", "pop_size": 1000, "core_size": 1200000, "pan_genes": 6000, "accessory_genes": 4000,
                   "selection": "prop_positive=0.1", "competition_strength": 0.5, "pairs": 100000},
        "cpu_baseline": {"value": val, "unit": "generations/s", "cores": threads, "kind": "port",
                         "sample": f"{steps_run} full cfg2 generations (oracle C port of population.rs, OpenMP over rows/pairs "
                                   f"where the reference uses rayon); distance pass on {pairs} pairs"},
        "distances": {"value": pairs_per_s, "unit": "pairs/s"},
        "e2e": {"value": val, "unit": "generations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=_JSON_OUT, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100, help="generations in the timed batch")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"],
                    help="reference: the CPU oracle port, --steps cfg2 generations at a few seconds each")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-gens", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=1, help="timed batches of --steps generations; the median batch is reported")
    ap.add_argument("--no-cfg4", action="store_true", help="skip the cfg4 strong-scaling record")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the state after the last timed generation as DIR/<name>.npy (rank 0's slab when N > 1)")
    args = ap.parse_args()
    if args.steps < 1 or args.repeats < 1:
        ap.error("--steps and --repeats must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; the reference arm has none")
    # stdout carries exactly ONE JSON line: libraries that print there (NCCL's version banner) are
    # sent to stderr, and the line is written to the saved descriptor at the end
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    # clocks / throttle reasons are sampled (every 100 ms) from here to the end of the end-to-end
    # loop: nvidia-smi needs ~1 s to start and the K-step region itself lasts tens of milliseconds
    sampler = ClockSampler(local_rank) if rank == 0 else None

    import torch
    import torch.distributed as dist
    import pansim_b200 as pb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; pansim_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    # diagnostics (tools/gpu_call_8d.sh): which ingredient of a multi-rank run changes the per-rank step time
    backend = os.environ.get("BENCH_DIST_BACKEND", "nccl")
    no_comm = os.environ.get("BENCH_NO_COMM") == "1"
    no_shard = os.environ.get("BENCH_NO_SHARD") == "1"
    fake_world, fake_rank = int(os.environ.get("BENCH_FAKE_WORLD", "0")), int(os.environ.get("BENCH_FAKE_RANK", "0"))
    if world > 1:
        if backend == "nccl":
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        else:
            dist.init_process_group(backend)
    red_dev = "cuda" if backend == "nccl" else "cpu"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=red_dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # batches of 8 or more generations launch the selection chain as CUDA graphs, one graph per phase of the
    # rotating buffers (6 phases), captured on first use: a warm-up of at least 8 keeps the captures out of
    # the timed batch
    W = max(8, args.warmup)
    K = args.steps
    R = args.repeats
    # this rank's slab: columns [rank*L, (rank+1)*L) of a (world*L)-site alignment
    from pansim_b200.sharding import SITE_ALIGN, ShardedPansim, broadcast_unique_id, column_shards
    L = CFG2["core_size"]
    cfg_world, cfg_rank = (fake_world, fake_rank) if fake_world else ((1, 0) if no_shard else (world, rank))
    Lslab = L if cfg_world == 1 else ((L + SITE_ALIGN - 1) // SITE_ALIGN) * SITE_ALIGN   # whole regions per rank
    total_L = L if cfg_world == 1 else Lslab * cfg_world
    kw = dict(CFG2)
    kw["core_size"] = total_L
    # Weak scaling = the same work on every rank. The per-site core rates of cfg2 are kept as the alignment
    # grows (lambda scales with its length, main.rs:275). The reference ties the HGT event count of the
    # ACCESSORY genome to the core mutation count (main.rs:280: round(n_core_mutations * HGT_rate)), so an
    # N-times longer alignment would also make the replicated accessory genome turn over N times faster and
    # its selection chain heavier on every rank (measured: 198 instead of 166 us per generation at N = 8,
    # profiles/r02_scaling_diag.md). HGT_rate / N keeps the accessory genome exactly cfg2's.
    kw["HGT_rate"] = pb.Params().HGT_rate / cfg_world
    p = pb.Params(**kw)
    d = pb.derive(p)

    # ---- multi-GPU parity, visible to the driver: a small column-sharded run must equal the unsharded one
    shard_parity = None
    if world > 1 and not (no_comm or no_shard):
        shard_parity = check_shard_parity(pb, ShardedPansim, rank, world, local_rank, dist, torch)

    site_begin, site_end = (0, 0) if cfg_world == 1 else column_shards(total_L, cfg_world)[cfg_rank]
    sim = pb.Pansim.from_params(p, device=local_rank, site_begin=site_begin, site_end=site_end)
    if world > 1 and not (no_comm or no_shard):
        sim.comm_init_rank(world, rank, broadcast_unique_id(rank))      # NCCL communicator inside the library
    info = sim.info()

    rng = np.random.default_rng(CFG2["seed"])           # identical on every rank
    sel = selection_coefficients(rng, d.pan_size, p.prop_positive)
    core_row = (1 << rng.integers(0, 4, total_L)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < d.avg_gene_freq_adj).astype(np.uint8)
    r1, r2 = sample_pairs(rng, p.pop_size, p.max_distances)
    sim.set_initial(core_row, acc_row)
    sim.set_selection(sel)

    def gather_ranks(x: float):
        if world == 1:
            return [x]
        t = torch.zeros(world, dtype=torch.float64, device=red_dev)
        t[rank] = x
        dist.all_reduce(t)
        return [float(v) for v in t.tolist()]

    # ---- warm-up (also diversifies the clonal start) -------------------------
    t_load0 = time.time()
    gen = 0
    sim.run_generations(gen, W)
    gen += W
    sim.pair_counts(r1, r2)

    # ---- timed region: device-resident, R batches of exactly K generations ----
    batch_ms, batch_rank_ms, wall_ms_list = [], [], []
    tm = None
    for _ in range(R):
        barrier()
        t0 = time.perf_counter()
        sim.run_generations(gen, K)             # K x (competition, fitness, parents, acc step, core step)
        tm = sim.timing()                        # synchronises the context's streams
        barrier()
        wall_ms_list.append(1e3 * (time.perf_counter() - t0))
        gen += K
        per_rank = gather_ranks(float(tm.total_ms))
        batch_rank_ms.append(per_rank)
        batch_ms.append(max(per_rank))           # max over ranks
    order = sorted(range(R), key=lambda i: batch_ms[i])
    med = order[R // 2]
    dev_ms = batch_ms[med]
    wall_ms = wall_ms_list[med]
    core_ms = float(tm.core_step_ms) / K            # last batch: core_mut_kernel (+ stand-alone recombination launches, if any)
    hr_ms = float(tm.core_hr_ms) / K                # stand-alone recombination launches: 0 in the deferred mode
    mut_ms = core_ms - hr_ms                        # core_mut_kernel: gather + deferred recombination + SNPs
    launches = int(tm.launches)
    select_ms, acc_ms = tm.select_ms / K, tm.acc_step_ms / K
    distinct_parents = int(len(np.unique(sim.parents())))      # rows the gather of the last generation actually read
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sim)
    if os.environ.get("BENCH_DIAG") == "1":        # diagnostics: the generation batches only
        if rank == 0:
            print(json.dumps({"diag": os.environ.get("BENCH_DIAG_NAME", ""), "world": world, "backend": backend, "no_comm": no_comm,
                              "no_shard": no_shard, "fake_world": fake_world, "site_begin": int(site_begin),
                              "us_per_step": 1e3 * dev_ms / K, "core_us": 1e3 * mut_ms, "select_us": 1e3 * select_ms,
                              "acc_us": 1e3 * acc_ms, "per_rank_us": [1e3 * x / K for x in batch_rank_ms[med]]}), file=_JSON_OUT, flush=True)
        sim.close()
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- distance pass (device time of the kernels; pairs resident; N > 1: + ncclAllReduce in the library) ----
    n_dist = max(3, min(10, K))
    pair_core_ms = pair_acc_ms = 0.0
    pair_total = []
    barrier()
    for _ in range(n_dist):
        sim.pair_counts(r1, r2)
        t = sim.timing()
        pair_core_ms += t.pair_core_ms
        pair_acc_ms += t.pair_acc_ms
        pair_total.append(float(t.total_ms))     # kernels + all-reduce, CUDA events on the library stream
    barrier()
    pair_ms = max_over_ranks(float(np.median(pair_total)))

    # ---- true cfg2: the step WITH its per-generation distance pass (main.rs:502-519) ----
    # recombination materialised for the reader every generation, mean / std on the device
    Kp = max(3, min(20, K))
    barrier()
    sim.run_generations_stats(gen, 2, r1, r2)
    gen += 2
    barrier()
    stats = sim.run_generations_stats(gen, Kp, r1, r2)
    tp = sim.timing()
    gen += Kp
    print_dist_ms = max_over_ranks(float(tp.total_ms)) / Kp

    # ---- end to end through the reference-facing API with HOST buffers --------
    # per generation the calls main.rs:435-464 makes, vectors crossing the boundary
    Ke = min(K, 50)
    e2e_runs = []
    for _ in range(5):
        barrier()
        t0 = time.perf_counter()
        for g in range(Ke):
            avg, parents = sim.select_parents(gen + g, reuse=True)   # average_distance + sample_indices: d2h N f64 + N u32
            sim.step_with_parents(gen + g, parents)            # h2d N u32
        barrier()
        e2e_runs.append(max_over_ranks(1e3 * (time.perf_counter() - t0) / Ke))
        gen += Ke
    e2e_ms = float(np.median(e2e_runs))
    t0 = time.perf_counter()
    for _ in range(3):
        cd, it, un = sim.pair_counts(r1, r2)               # h2d 2 x P u32 (first call), d2h 3 x P u32
    e2e_pair_ms = 1e3 * (time.perf_counter() - t0) / 3
    t0 = time.perf_counter()
    for _ in range(3):
        st1 = sim.pair_stats(r1, r2)                       # d2h 4 f64
    e2e_stats_ms = 1e3 * (time.perf_counter() - t0) / 3
    # --print_matrices: _core_genome.csv (2 bytes of text per site) expanded on the GPU and streamed through
    # two pinned chunks; /dev/null as the file takes the disk out of the number (PCIe + the pipeline remain)
    export = None
    if world == 1 and rank == 0:
        sim.write_core_csv("/dev/null")
        t0 = time.perf_counter()
        nbytes = sim.write_core_csv("/dev/null")
        dt = time.perf_counter() - t0
        export = {"bytes": int(nbytes), "seconds": dt, "GBps": nbytes / dt / 1e9,
                  "what": "pansim_write_core_csv to /dev/null: text expansion kernel + device-to-host copies of 32 MB pinned chunks, "
                          "double buffered (population.rs:877-879 builds the same text with to_string + join per element)"}
    clocks = sampler.stop(t_load0, time.time()) if sampler else None
    sim.close()

    # ---- cfg4: strong scaling of the SAME 10 000 x 5 Mbp x 18 000 problem over the ranks ----
    cfg4 = None
    if not args.no_cfg4:
        cfg4 = run_cfg4_strong(pb, rank, world, local_rank, barrier, max_over_ranks, gather_ranks,
                               column_shards, broadcast_unique_id)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    N, P = p.pop_size, p.max_distances
    core_bytes = 2 * N * ((info.local_sites + 3) // 4)              # read + write of the packed slab
    achieved = core_bytes / (mut_ms * 1e-3) / 1e9 if mut_ms > 0 else 0.0
    gen_bytes = int(info.algorithmic_bytes_per_generation)
    ms_per_step = dev_ms / K
    value = world * K / (dev_ms * 1e-3)
    pair_bytes = int(info.algorithmic_bytes_per_pair)
    pairs_per_s = world * P / (pair_ms * 1e-3)
    tr_core = ncu_traffic("core_mut_kernel")
    tr_pair = ncu_traffic("pair_core_kernel")
    words_per_pair = (info.local_sites + 15) // 16 + 2 * ((d.pan_size + 31) // 32)      # SURVEY.md 8d: 32-bit word-compares
    popc_peak = 16 * 148 * 1.965e9                                                    # POPC: 16 / clk / SM at 1965 MHz
    compulsory = N * ((info.local_sites + 3) // 4 + (d.pan_size + 7) // 8)

    line = {
        "metric": "generations/sec", "value": value, "unit": "generations/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "cfg2", "pop_size": N, "core_size": int(info.local_sites), "pan_genes": p.pan_genes,
                   "accessory_genes": d.pan_size, "selection": "prop_positive=0.1",
                   "competition_strength": p.competition_strength, "pairs": P,
                   "core_size_per_gpu": int(info.local_sites),
                   "sharding": "columns; accessory replicated; no collective in the generation step; "
                               "distance pass: ncclAllReduce of the core counts inside the library",
                   "weak_scaling": "every rank holds a cfg2 slab (1.2 Mbp x 1000) of an N x 1.2 Mbp alignment; per-site core rates "
                                   "and the accessory genome's event counts are cfg2's at every N (HGT_rate / N, because "
                                   "main.rs:280 ties the HGT count to the alignment length)",
                   "l2": "inputs larger than L2 (2 x %.0f MB packed state, double buffered)" % (info.core_state_bytes / 1e6),
                   "timing": "CUDA events on the library stream around each batch of K generations, max over ranks, "
                             "median of the R batches"},
        "repeats": {"n": R, "ms_per_step_min": min(batch_ms) / K, "ms_per_step_median": dev_ms / K,
                    "ms_per_step_max": max(batch_ms) / K, "busy_ms": sum(batch_ms),
                    "per_rank_ms_per_step_median_batch": [x / K for x in batch_rank_ms[med]]},
        "wall_ms_per_step": wall_ms / K,
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"kernel": "core_mut_kernel<RNG> (gather-by-parent + previous generation's recombination events + SNP "
                               "mutation in one pass, TMA bulk pipeline)",
                     "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak,
                     "traffic": (tr_core["dram_read_bytes"] + tr_core["dram_write_bytes"]) if tr_core else None,
                     "traffic_source": tr_core["source"] if tr_core else None,
                     "traffic_note": "gather-by-parent reads every DISTINCT parent row from DRAM once, the children of the same parent "
                                     "hit in L2: with cfg2's selection + competition only %d of %d individuals were parents in the last "
                                     "generation, so the read side is far below the 300 MB of algorithmic reads; the neutral control "
                                     "(profiles/r02_l2_core_mut_rng.csv, ~630 distinct parents) reads 528 MB" % (distinct_parents, N),
                     "distinct_parents_last_generation": distinct_parents,
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": core_bytes, "launch_ms": mut_ms,
                     "core_genome_frac": core_bytes / (core_ms * 1e-3) / 1e9 / peak if core_ms > 0 else None,
                     "step_algorithmic_bytes": gen_bytes,
                     "step_frac": gen_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                     "kernel_share_of_step": mut_ms / ms_per_step if ms_per_step > 0 else None,
                     "breakdown_ms": {"select": select_ms, "acc_step": acc_ms, "core_step": core_ms,
                                      "core_mut": mut_ms, "core_hr": hr_ms}},
        "distances": {"value": pairs_per_s, "unit": "pairs/s", "ms_per_pass": pair_ms, "pairs": P,
                      "core_ms": pair_core_ms / n_dist, "acc_ms": pair_acc_ms / n_dist,
                      "streaming_GBps": pair_bytes * P / (pair_ms * 1e-3) / 1e9,
                      "streaming_frac_of_hbm_peak": pair_bytes * P / (pair_ms * 1e-3) / 1e9 / peak,
                      "word_compares_per_pair": words_per_pair,
                      "popc_pipe_frac": (P / (pair_ms * 1e-3)) * words_per_pair / popc_peak,
                      "popc_pipe_note": "SURVEY.md 8d model: one POPC per 32-bit word-compare at 16 POPC/clk/SM. The plane-form kernels "
                                        "count 64 sites (4 words) with ONE POPC (carry-save), so this fraction can exceed 1; the model that "
                                        "bounds them is the ALU pipe: per 64 sites 4 LOP3 (masks) + 2 LOP3 (carry-save) + 1 POPC (a quarter "
                                        "of the LOP3 rate = 4 slots) + 1 IADD = 11 slots at 64 slots/clk/SM",
                      "alu_slots_per_64_sites": 11,
                      "alu_model_frac": (P / (pair_ms * 1e-3)) * ((info.local_sites + 63) // 64) * 11 / (64 * 148 * 1.965e9),
                      "thread_instructions_per_word_compare": (tr_pair["warp_instructions"] * 32 / (P * words_per_pair)) if tr_pair else None,
                      "compulsory_dram_bytes": compulsory,
                      "dram_bytes_per_pass": (tr_pair["dram_read_bytes"] + tr_pair["dram_write_bytes"]) if tr_pair else None,
                      "dram_over_compulsory": ((tr_pair["dram_read_bytes"] + tr_pair["dram_write_bytes"]) / compulsory) if tr_pair else None,
                      "dram_source": tr_pair["source"] if tr_pair else None,
                      "e2e_pairs_per_s": P / (e2e_pair_ms * 1e-3),
                      "e2e_h2d_bytes": 0, "e2e_d2h_bytes": 12 * P,
                      "e2e_note": "pair list unchanged since the previous call: validated and uploaded once (8 x P bytes), then cached",
                      "e2e_stats_ms": e2e_stats_ms, "e2e_stats_d2h_bytes": 32},
        "cfg2_print_dist": {"value": world / (print_dist_ms * 1e-3), "unit": "generations/s", "ms_per_generation": print_dist_ms,
                            "generations": Kp, "d2h_bytes_per_generation": 32,
                            "what": "pansim_run_generations_stats: generation step + recombination materialised + distance pass over "
                                    "%d pairs + mean/std on the device, every generation (main.rs:435-519 with --print_dist)" % P,
                            "last_stats": [float(x) for x in stats[-1]]},
        "e2e": {"value": world / (e2e_ms * 1e-3), "unit": "generations/s",
                "h2d_bytes_per_step": 4 * N, "d2h_bytes_per_step": 12 * N, "ms_per_step": e2e_ms,
                "runs_ms_per_step": e2e_runs,
                "path": "pansim_select_parents (average_distance + sample_indices, one read-back) -> pansim_step_with_parents, "
                        "host vectors; the step call returns with the core kernel in flight, each run ends with a device synchronize"},
    }
    if export is not None:
        line["export_core_csv"] = export
    if shard_parity is not None:
        line["shard_parity"] = bool(shard_parity)
    if cfg4 is not None:
        line["cfg4_strong"] = cfg4
    if not args.no_cpu_baseline and world == 1:
        pairs_cpu = 2000
        threads, t_gen, t_dist = cpu_baseline_sample(args.cpu_gens, True, pairs_cpu)
        line["cpu_baseline"] = {
            "value": args.cpu_gens / t_gen, "unit": "generations/s", "cores": threads, "kind": "port",
            "sample": f"{args.cpu_gens} cfg2 generations from the clonal start (oracle C port, OpenMP where the "
                      f"reference uses rayon); distance pass on {pairs_cpu} of the pairs",
            "distances_pairs_per_s": args.cpu_gens * pairs_cpu / t_dist if t_dist > 0 else None}
    print(json.dumps(line), file=_JSON_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()
    if shard_parity is False:
        raise SystemExit("bench.py: column-sharded run differs from the unsharded run (shard_parity false)")


def dump_outputs(out_dir: str, sim) -> None:
    """--dump-outputs: what a caller of run_generations holds after the last timed generation (about 33 MB
    at cfg2). The core state (N x 1.2 Mbp one-hot bytes) is too large to store whole, so a fixed, seeded
    sample of 4096 sites of every row is written, and every row's A / C / G / T counts over all sites
    show a change anywhere in the row."""
    os.makedirs(out_dir, exist_ok=True)
    core = sim.download_core()
    sites = np.sort(np.random.default_rng(1).choice(core.shape[1], size=min(4096, core.shape[1]), replace=False))
    arrays = {
        "parents": sim.parents().astype(np.float64),
        "acc": sim.download_acc().astype(np.float32),
        "core_sample": core[:, sites].astype(np.float32),
        "core_sample_sites": sites.astype(np.float64),
        "core_allele_counts": np.stack([np.bincount(row, minlength=9)[[1, 2, 4, 8]] for row in core]).astype(np.float64),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def check_shard_parity(pb, ShardedPansim, rank, world, local_rank, dist, torch) -> bool:
    """tests/multi_gpu_worker.py in short: sharded state, parents, all-reduced pair counts and
    on-device statistics equal those of an unsharded context on the same device."""
    p = pb.Params(pop_size=96, core_size=8192 * 9 + 123, pan_genes=700, core_genes=200, n_gen=3, max_distances=400,
                  seed=5, prop_positive=0.1, competition_strength=0.3, HR_rate=0.5)
    d = pb.derive(p)
    rng = np.random.default_rng(1)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < 0.25).astype(np.uint8)
    sel = rng.normal(0, 0.05, d.pan_size)
    r1, r2 = sample_pairs(rng, p.pop_size, p.max_distances)
    sh = ShardedPansim(p, rank, world, device=local_rank)
    whole = pb.Pansim.from_params(p, device=local_rank)
    for s in (sh, whole):
        s.set_initial(core_row, acc_row)
        s.set_selection(sel)
        s.run_generations(0, p.n_gen)
    b, e = sh.shards[rank]
    ok = all((x == y).all() for x, y in zip(sh.pair_counts(r1, r2), whole.pair_counts(r1, r2)))
    ok = ok and (sh.download_acc() == whole.download_acc()).all() and (sh.parents() == whole.parents()).all()
    ok = ok and (sh.download_core() == whole.download_core()[:, b:e]).all()
    ok = ok and sh.pair_stats(r1, r2) == whole.pair_stats(r1, r2)
    sh.sim.close()
    whole.close()
    t = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return int(t.item()) == 1


def run_cfg4_strong(pb, rank, world, local_rank, barrier, max_over_ranks, gather_ranks, column_shards, broadcast_unique_id):
    """BASELINE configs[3]: pop_size 10 000, core 5 Mbp, 20 000 pan genes (18 000 accessory), defaults
    otherwise (neutral, no competition), column-sharded over the ranks: STRONG scaling, every N runs
    the same problem. Reports ms per generation (max over ranks) and the pieces that do not shrink."""
    import torch
    kw = dict(pop_size=10_000, core_size=5_000_000, pan_genes=20_000, core_genes=2_000, n_gen=500, max_distances=20_000, seed=0)
    p = pb.Params(**kw)
    d = pb.derive(p)
    b, e = (0, 0) if world == 1 else column_shards(p.core_size, world)[rank]
    try:
        sim = pb.Pansim.from_params(p, device=local_rank, site_begin=b, site_end=e)
    except Exception as ex:            # e.g. not enough memory beside another tenant
        return {"error": str(ex)[:200]} if rank == 0 else None
    if world > 1:
        sim.comm_init_rank(world, rank, broadcast_unique_id(rank))
    rng = np.random.default_rng(0)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < d.avg_gene_freq_adj).astype(np.uint8)
    r1, r2 = sample_pairs(rng, p.pop_size, p.max_distances)
    sim.set_initial(core_row, acc_row)
    sim.set_selection(np.zeros(d.pan_size))
    sim.run_generations(0, 3)
    G = 10
    runs = []
    tm = None
    for rep in range(3):
        barrier()
        sim.run_generations(3 + rep * G, G)
        tm = sim.timing()
        barrier()
        runs.append(max(gather_ranks(float(tm.total_ms))) / G)
    ms = float(np.median(runs))
    core_ms = max_over_ranks(float(tm.core_step_ms) / G)
    select_ms = max_over_ranks(float(tm.select_ms) / G)
    acc_ms = max_over_ranks(float(tm.acc_step_ms) / G)
    sim.pair_counts(r1, r2)
    barrier()
    sim.pair_counts(r1, r2)
    tp = sim.timing()
    pair_ms = max_over_ranks(float(tp.total_ms))
    info = sim.info()
    sim.close()
    peak, _ = measured_peak()
    total_bytes = 2 * p.pop_size * ((p.core_size + 3) // 4) + 2 * p.pop_size * ((d.pan_size + 7) // 8)
    return {"workload": "cfg4", "pop_size": p.pop_size, "core_size": p.core_size, "accessory_genes": d.pan_size,
            "n_gpus": world, "scaling": "strong", "generations": G, "ms_per_generation": ms, "runs_ms": runs,
            "generations_per_s": 1e3 / ms, "local_sites": int(info.local_sites),
            "hbm_frac_all_gpus": total_bytes / (ms * 1e-3) / 1e9 / (peak * world),
            "core_step_ms": core_ms, "replicated_chain_ms": {"select": select_ms, "acc_step": acc_ms},
            "note": "the selection chain and the accessory step are replicated on every rank (they do not shrink with N); "
                    "they run on their own streams beside the core step",
            "pairs": p.max_distances, "pair_pass_ms_incl_allreduce": pair_ms,
            "pairs_per_s": p.max_distances / (pair_ms * 1e-3)}


if __name__ == "__main__":
    main()
