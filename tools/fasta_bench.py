"""Timing of the core-genome FASTA export (pansim_b200/csrc/fasta.cuh), one GPU call.

  python tools/fasta_bench.py [--out profiles/r07_fasta_bench.json] [--reps 5] [--kernel_reps 10]

Three shapes, each evolved on the device from a clonal start (no one-hot upload from the host):
  cfg1        1 000 x 1.2 Mbp,  3 generations at the default rates: every site polymorphic (~1.2 GB of FASTA)
  cfg1_sparse 1 000 x 1.2 Mbp, 20 generations at core_mu 1e-6 (two SNPs per genome per generation): few columns
  cfg1_10k   10 000 x 1.2 Mbp,  3 generations at the default rates (~12 GB of FASTA)
For each shape and both modes (whole: every site; snps: the polymorphic columns):
  - kernel time from the library's CUDA events (pansim_core_fasta_kernel_ms): the site pass (SNP mode only: allele
    counts, polymorphic sites, scan, column list; whole mode has none, reported as null) and the expansion of every
    chunk of records into device memory, mean of --kernel_reps after a warm-up;
  - the expansion's bytes, the packed words that hold a column (4 bytes each, once per row: every word of the row in
    whole mode, only the words of polymorphic sites in SNP mode) plus the text written, over its kernel time,
    against the measured HBM copy bandwidth of 6 529 GB/s (BASELINE.md);
  - end to end: pansim_write_core_fasta in both modes and pansim_write_core_csv of the same state to /dev/null,
    wall time around each call (all synchronise), the three arms alternated, median of --reps.
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

HBM_GBS = 6529.1                # measured HBM copy (BASELINE.md)
SHAPES = [("cfg1", 1000, 1_200_000, 3, None), ("cfg1_sparse", 1000, 1_200_000, 20, 1e-6),
          ("cfg1_10k", 10_000, 1_200_000, 3, None)]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def case(name, N, L, gens, core_mu, reps, kernel_reps):
    kw = {} if core_mu is None else {"core_mu": core_mu}
    p = pb.Params(pop_size=N, core_size=L, pan_genes=600, core_genes=200, seed=1, **kw)
    d = pb.derive(p)
    rng = np.random.default_rng(1)
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial((1 << rng.integers(0, 4, L)).astype(np.uint8), (rng.random(d.pan_size) < 0.5).astype(np.uint8))
        sim.run_generations(0, gens)
        segregating = sim.core_diversity().segregating
        counts = sim.core_allele_counts()
        poly_words = len(np.unique(np.flatnonzero((counts > 0).sum(axis=1) >= 2) // 16))
        kernels = {}
        for mode, snps in (("whole", False), ("snps", True)):
            site_ms, expand_ms, text = sim.fasta_kernel_ms(snps, kernel_reps)
            read = N * (poly_words if snps else (L + 15) // 16) * 4
            gbs = (read + text) / (expand_ms * 1e-3) / 1e9 if expand_ms else None
            kernels[mode] = {"reps": kernel_reps, "site_pass_ms": site_ms if snps else None, "expansion_ms": expand_ms,
                             "text_bytes": text, "words_read_per_row": poly_words if snps else (L + 15) // 16,
                             "expansion_bytes": read + text, "expansion_gbs": gbs,
                             "expansion_frac_of_hbm": gbs / HBM_GBS if gbs else None}
        arms = {"whole": lambda: sim.write_core_fasta("/dev/null").bytes,
                "snps": lambda: sim.write_core_fasta("/dev/null", snps_only=True).bytes,
                "csv": lambda: sim.write_core_csv("/dev/null")}
        snp = sim.write_core_fasta("/dev/null", snps_only=True)
        sizes = {k: f() for k, f in arms.items()}                                   # warm-up
        times = {k: [] for k in arms}
        for _ in range(reps):
            for k, f in arms.items():
                t = time.perf_counter()
                f()
                times[k].append(time.perf_counter() - t)
    med = {k: statistics.median(v) for k, v in times.items()}
    gbs = {k: sizes[k] / med[k] / 1e9 for k in med}
    return {"config": name, "pop_size": N, "core_size": L, "state": f"{gens} generations from a clonal start"
            + ("" if core_mu is None else f" at core_mu {core_mu}"), "segregating": segregating,
            "snp_columns": snp.columns, "const_counts": [int(x) for x in snp.const_counts], "kernels": kernels,
            "end_to_end": {"reps": reps, "file_bytes": sizes, "median_s": med, "all_s": times, "gbs": gbs,
                           "whole_over_csv_time": med["whole"] / med["csv"], "snps_over_csv_time": med["snps"] / med["csv"],
                           "kernels_share_of_whole": kernels["whole"]["expansion_ms"] * 1e-3 / med["whole"],
                           "kernels_share_of_snps": (kernels["snps"]["site_pass_ms"] + kernels["snps"]["expansion_ms"]) * 1e-3 / med["snps"]}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--kernel_reps", type=int, default=10)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    args = ap.parse_args()
    want = args.shapes.split(",")
    res = {"gpu": gpu_info(), "hbm_gbs_reference": HBM_GBS,
           "cases": [case(*s, args.reps, args.kernel_reps) for s in SHAPES if s[0] in want]}
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
