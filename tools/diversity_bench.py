"""Timing of the core-genome diversity reduction (pansim_b200/csrc/diversity.cuh), one GPU call.

  python tools/diversity_bench.py [--out profiles/r03_diversity_bench.json] [--reps 20] [--gens 40]

1. pansim_core_diversity without and with the SFS at cfg1 (1 000 x 1.2 Mbp) and cfg4 (10 000 x 5 Mbp): kernel time
   from the library's CUDA events (pansim_get_timing total_ms after the call), median and minimum of --reps calls.
   The packed state (300 MB, 12.5 GB) is larger than the 126 MB L2, and every call streams it from the first row to
   the last, so the passes read HBM. Achieved GB/s counts the algorithmic bytes N * ceil(L/16) * 4.
   cfg1 holds uniformly random rows (every site segregating: the most SFS atomics); cfg4 starts clonal and runs
   --cfg4_gens generations at the default rates (the JSON records how many sites segregate).
2. The batch at cfg2 (bench.py's workload): microseconds per generation of run_generations against
   run_generations_diversity without pairs, and of run_generations_stats against run_generations_diversity with the
   100 000 sampled pairs; wall time around each (synchronising) call, arms alternated, median of --batch_reps.
The card name and power limit are read with `nvidia-smi --query-gpu=name,power.limit --format=csv` in the same call.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import pansim_b200 as pb  # noqa: E402

PEAK_FALLBACK_GBS = 6650.0      # the figure bench.py uses without MEASURED_PEAKS.json
CFG2 = dict(pop_size=1000, core_size=1_200_000, pan_genes=6000, core_genes=2000, n_gen=100,
            max_distances=100_000, prop_positive=0.1, competition_strength=0.5, seed=0)


def peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return PEAK_FALLBACK_GBS, "bench.py fallback (no MEASURED_PEAKS.json)"


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def time_reduction(sim, sfs, reps):
    sim.core_diversity(sfs=sfs)                 # warm-up (module load, buffers)
    ms = []
    for _ in range(reps):
        sim.core_diversity(sfs=sfs)
        ms.append(sim.timing().total_ms)
    return ms


def reduction_case(name, N, L, reps, peak, state):
    p = pb.Params(pop_size=N, core_size=L, pan_genes=600, core_genes=200, seed=1)
    rng = np.random.default_rng(1)
    d = pb.derive(p)
    out = {}
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial((1 << rng.integers(0, 4, L)).astype(np.uint8), (rng.random(d.pan_size) < 0.5).astype(np.uint8))
        if state == "random":
            sim.upload(np.left_shift(np.uint8(1), rng.integers(0, 4, (N, L), dtype=np.uint8)))
        else:
            sim.run_generations(0, state)
        div, sfs = sim.core_diversity(sfs=True)
        bytes_alg = N * ((L + 15) // 16) * 4
        for with_sfs in (False, True):
            ms = time_reduction(sim, with_sfs, reps)
            med = statistics.median(ms)
            gbs = bytes_alg / (med * 1e-3) / 1e9
            out["sfs" if with_sfs else "no_sfs"] = {
                "median_us": med * 1e3, "min_us": min(ms) * 1e3, "reps": reps,
                "achieved_gbs": gbs, "achieved_gbs_at_min": bytes_alg / (min(ms) * 1e-3) / 1e9, "frac_of_hbm": gbs / peak}
    return {"config": name, "pop_size": N, "core_size": L, "algorithmic_bytes": bytes_alg,
            "state": "uniformly random rows" if state == "random" else f"{state} generations from a clonal start",
            "segregating": div.segregating, "multiallelic": div.multiallelic, "nonzero_sfs_bins": int((sfs > 0).sum()), **out}


def batch_case(gens, reps):
    p = pb.Params(**CFG2)
    d = pb.derive(p)
    rng = np.random.default_rng(0)
    sel = rng.normal(0, 0.05, d.pan_size)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < d.avg_gene_freq_adj).astype(np.uint8)
    r1 = rng.integers(0, p.pop_size, p.max_distances).astype(np.uint32)
    r2 = rng.integers(0, p.pop_size - 1, p.max_distances).astype(np.uint32)
    r2 = (r2 + (r2 >= r1)).astype(np.uint32)
    arms = {
        "run_generations": lambda s, g0: s.run_generations(g0, gens),
        "run_generations_diversity": lambda s, g0: s.run_generations_diversity(g0, gens),
        "run_generations_stats": lambda s, g0: s.run_generations_stats(g0, gens, r1, r2),
        "run_generations_diversity_pairs": lambda s, g0: s.run_generations_diversity(g0, gens, r1, r2),
    }
    times = {k: [] for k in arms}
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(sel)
        g0 = 0
        for f in arms.values():                  # warm-up: graphs captured, buffers sized
            f(sim, g0)
            g0 += gens
        for _ in range(reps):
            for k, f in arms.items():
                t = time.perf_counter()
                f(sim, g0)
                times[k].append((time.perf_counter() - t) * 1e6 / gens)
                g0 += gens
    med = {k: statistics.median(v) for k, v in times.items()}
    return {"config": "cfg2", "generations_per_call": gens, "reps": reps,
            "us_per_generation_median": med, "us_per_generation_all": times,
            "diversity_overhead_us": med["run_generations_diversity"] - med["run_generations"],
            "diversity_overhead_with_pairs_us": med["run_generations_diversity_pairs"] - med["run_generations_stats"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--gens", type=int, default=40)
    ap.add_argument("--batch_reps", type=int, default=5)
    ap.add_argument("--cfg4_gens", type=int, default=3)
    args = ap.parse_args()
    peak, peak_src = peak_gbs()
    res = {"gpu": gpu_info(), "hbm_gbs_reference": peak, "hbm_reference_source": peak_src,
           "reduction": [reduction_case("cfg1", 1000, 1_200_000, args.reps, peak, "random"),
                         reduction_case("cfg4", 10_000, 5_000_000, args.reps, peak, args.cfg4_gens)],
           "batch": batch_case(args.gens, args.batch_reps)}
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
