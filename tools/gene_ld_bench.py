"""Timing of the accessory-gene linkage pass (pansim_b200/csrc/gene_ld.cuh), one GPU call.

  python tools/gene_ld_bench.py [--out profiles/r08_gene_ld_bench.json] [--reps 5] [--kernel_reps 10]

Shapes, each evolved on the device from a clonal start (every row the same random accessory row, so every gene
starts fixed), at the low flip rates --rate_genes1 1e-4 --rate_genes2 1e-2 with --HGT_rate 0.05:
  cfg1        1 000 x G 4 000,  300 generations
  cfg4_acc   10 000 x G 18 000, 100 generations (a 10 kbp core: only the accessory matrix is read)
  cfg5_acc   20 000 x G 4 000,  100 generations
and a control, cfg1 at the default rates (1 and 1 000 hits per gene compartment and generation), 50 generations.
For each:
  - kernel times from the library's CUDA events (pansim_gene_ld_kernel_ms), mean of --kernel_reps after a warm-up:
    the gene pass (presence counts, used genes, scan, compaction), the transpose to bit rows, the pair pass (zeroed
    outputs and pair kernel);
  - pairs per second of the pair pass; the i8 tensor rate 2 K 128^2 tile_pairs / pair time (K = rows padded to the
    MMA step) against the data sheet's dense INT8 rate of a B200, 4 500 TOPS (a data-sheet figure, not a measurement);
  - end to end: pansim_gene_ld, wall time around the call (it synchronises), median of --reps;
  - what the state shows per class: pairs, mean r^2, associated / dissociated / four-gamete shares, used genes.
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

INT8_TOPS_DATASHEET = 4500.0    # B200 dense INT8, data sheet (72 POPS for eight GPUs with sparsity / 16)
LOW = dict(rate_genes1=1e-4, rate_genes2=1e-2, HGT_rate=0.05)
SHAPES = [("cfg1", 1000, 6000, 2000, 300, LOW), ("cfg4_acc", 10_000, 20_000, 2000, 100, LOW),
          ("cfg5_acc", 20_000, 6000, 2000, 100, LOW), ("cfg1_default_rates", 1000, 6000, 2000, 50, {})]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def case(name, N, pan_genes, core_genes, gens, rates, reps, kernel_reps, r2_bins):
    p = pb.Params(pop_size=N, core_size=10_000, pan_genes=pan_genes, core_genes=core_genes, seed=1, **rates)
    d = pb.derive(p)
    rng = np.random.default_rng(1)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, (rng.random(d.pan_size) < 0.5).astype(np.uint8))
        sim.run_generations(0, gens)
        gene_ms, tr_ms, pair_ms, pairs = sim.gene_ld_kernel_ms(r2_bins, 1, kernel_reps)
        res = sim.gene_ld(r2_bins)                                  # warm-up of the end-to-end call
        assert int(res.pairs.sum()) == pairs
        times = []
        for _ in range(reps):
            t = time.perf_counter()
            sim.gene_ld(r2_bins)
            times.append(time.perf_counter() - t)
    used = int(res.genes_used.sum())
    n_t = -(-used // 128)
    tiles = n_t * (n_t + 1) // 2
    kw = -(-N // 64) * 2
    ops = 2 * kw * 32 * 128 * 128 * tiles
    med = statistics.median(times)
    return {
        "config": name, "pop_size": N, "genes": d.pan_size, "compartments": d.comp, "rates": rates,
        "state": f"{gens} generations from a clonal start", "genes_used": [int(x) for x in res.genes_used],
        "pairs": pairs, "tile_pairs": tiles,
        "kernels": {"reps": kernel_reps, "gene_pass_ms": gene_ms, "transpose_ms": tr_ms, "pair_pass_ms": pair_ms,
                    "pairs_per_s": pairs / (pair_ms * 1e-3) if pair_ms else None,
                    "i8_tensor_tops": ops / (pair_ms * 1e-3) / 1e12 if pair_ms else None,
                    "i8_frac_of_datasheet_dense": ops / (pair_ms * 1e-3) / 1e12 / INT8_TOPS_DATASHEET if pair_ms else None},
        "end_to_end": {"reps": reps, "median_ms": med * 1e3, "all_ms": [t * 1e3 for t in times], "pairs_per_s": pairs / med},
        "classes": {label: {"pairs": int(res.pairs[k]), "mean_r2": float(res.mean_r2[k]),
                            "associated_share": int(res.associated[k]) / max(1, int(res.pairs[k])),
                            "dissociated_share": int(res.dissociated[k]) / max(1, int(res.pairs[k])),
                            "four_gamete_share": int(res.four_gamete[k]) / max(1, int(res.pairs[k])),
                            "hist": [int(x) for x in res.hist[k]]}
                    for k, label in enumerate(res.classes)},
        "r2_floor_1_over_n": 1.0 / N}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--kernel_reps", type=int, default=10)
    ap.add_argument("--r2_bins", type=int, default=20)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    args = ap.parse_args()
    want = args.shapes.split(",")
    res = {"gpu": gpu_info(), "int8_tops_datasheet_dense": INT8_TOPS_DATASHEET, "cases": []}
    for s in SHAPES:
        if s[0] in want:
            res["cases"].append(case(*s, args.reps, args.kernel_reps, args.r2_bins))
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
