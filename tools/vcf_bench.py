"""Timing of the core-genome VCF export (pansim_b200/csrc/vcf.cuh), one GPU call.

  python tools/vcf_bench.py [--out profiles/r04_vcf_bench.json] [--reps 5] [--kernel_reps 10]

Three shapes, each evolved on the device from a clonal start (no one-hot upload from the host):
  cfg1        1 000 x 1.2 Mbp,  3 generations at the default rates: nearly every site is written (~2.4 GB of text)
  cfg1_sparse 1 000 x 1.2 Mbp, 20 generations at core_mu 1e-6 (two SNPs per genome per generation): few lines
  cfg1_10k   10 000 x 1.2 Mbp,  3 generations at the default rates (~24 GB of text, 40 row blocks per tile)
For each shape:
  - kernel time from the library's CUDA events (pansim_core_vcf_kernel_ms): the site pass (allele counts,
    descriptors, offset scan, chunking) and the expansion of every chunk into device memory, mean of --kernel_reps;
  - the expansion's bytes, N * ceil(L/16) * 4 read plus the text written, over its kernel time, against the
    measured HBM copy bandwidth of 6 529 GB/s (BASELINE.md);
  - end to end: pansim_write_core_vcf and pansim_write_core_csv of the same state to /dev/null, wall time around
    each call (both synchronise), the two arms alternated, median of --reps.
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
        _, sfs = sim.core_diversity(sfs=True)
        lines = L - int(sfs[0])
        site_ms, expand_ms, text = sim.vcf_kernel_ms(kernel_reps)
        read = N * ((L + 15) // 16) * 4
        times = {"vcf": [], "csv": []}
        sizes = {"vcf": sim.write_core_vcf("/dev/null"), "csv": sim.write_core_csv("/dev/null")}   # warm-up
        for _ in range(reps):
            for arm, f in (("vcf", lambda: sim.write_core_vcf("/dev/null")), ("csv", lambda: sim.write_core_csv("/dev/null"))):
                t = time.perf_counter()
                f()
                times[arm].append(time.perf_counter() - t)
    med = {k: statistics.median(v) for k, v in times.items()}
    gbs = {k: sizes[k] / med[k] / 1e9 for k in med}
    return {"config": name, "pop_size": N, "core_size": L, "state": f"{gens} generations from a clonal start"
            + ("" if core_mu is None else f" at core_mu {core_mu}"), "lines": lines, "fraction_of_sites_written": lines / L,
            "text_bytes": text,
            "kernels": {"reps": kernel_reps, "site_pass_ms": site_ms, "expansion_ms": expand_ms,
                        "expansion_bytes": read + text, "expansion_gbs": (read + text) / (expand_ms * 1e-3) / 1e9 if expand_ms else None,
                        "expansion_frac_of_hbm": (read + text) / (expand_ms * 1e-3) / 1e9 / HBM_GBS if expand_ms else None},
            "end_to_end": {"reps": reps, "file_bytes": sizes, "median_s": med, "all_s": times, "gbs": gbs,
                           "vcf_over_csv_gbs": gbs["vcf"] / gbs["csv"],
                           "kernels_share_of_vcf": (site_ms + expand_ms) * 1e-3 / med["vcf"],
                           "expansion_share_of_vcf": expand_ms * 1e-3 / med["vcf"]}}


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
