"""Timing of the core-genome LD pass (pansim_b200/csrc/ld.cuh), one GPU call.

  python tools/ld_bench.py [--out profiles/r05_ld_bench.json] [--reps 5] [--kernel_reps 10]

Three shapes, each evolved on the device from a clonal start:
  cfg1        1 000 x 1.2 Mbp,  3 generations at the default rates: nearly every site is used
  cfg1_sparse 1 000 x 1.2 Mbp, 20 generations at core_mu 1e-6: few used sites
  cfg1_10k   10 000 x 1.2 Mbp,  3 generations at the default rates
each with (max_dist, bin_width) = (10 000, 100) and (1 000, 10). For each:
  - kernel times from the library's CUDA events (pansim_core_ld_kernel_ms), mean of --kernel_reps after a warm-up:
    the site pass (allele counts, used sites, scan, compaction), the transpose to bit rows, the pair pass (tile list
    and pair kernel);
  - the transpose's bytes, N * ceil(L/16) * 4 read plus used * kw * 4 written, over its time, against the measured HBM
    copy bandwidth of 6 529 GB/s (BASELINE.md);
  - pairs per second of the pair pass; the share of the tile-pair work that falls inside the window (pairs over
    tile pairs x 128^2 / 2 on diagonal tiles, 128^2 elsewhere); the i8 tensor rate 2 K 128^2 tile_pairs / pair time
    (K = rows padded to the MMA step) against the data sheet's dense INT8 rate of a B200, 4 500 TOPS (a data-sheet
    figure, not a measurement);
  - end to end: pansim_core_ld, wall time around the call (it synchronises), median of --reps.
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
INT8_TOPS_DATASHEET = 4500.0    # B200 dense INT8, data sheet (72 POPS for eight GPUs with sparsity / 16)
SHAPES = [("cfg1", 1000, 1_200_000, 3, None), ("cfg1_sparse", 1000, 1_200_000, 20, 1e-6),
          ("cfg1_10k", 10_000, 1_200_000, 3, None)]
WINDOWS = [(10_000, 100), (1_000, 10)]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def tile_pairs(pos, max_dist):
    """Tile pairs and diagonal tile pairs of the pair kernel (ld_tiles_kernel), from the used-site positions."""
    U = len(pos)
    n_i = -(-U // 128)
    last = np.minimum((np.arange(n_i) + 1) * 128, U) - 1
    end = np.searchsorted(pos, pos[last] + max_dist, side="right") - 1
    return int((end // 128 - np.arange(n_i) + 1).sum()), n_i


def case(name, N, L, gens, core_mu, reps, kernel_reps):
    kw_ = {} if core_mu is None else {"core_mu": core_mu}
    p = pb.Params(pop_size=N, core_size=L, pan_genes=600, core_genes=200, seed=1, **kw_)
    d = pb.derive(p)
    rng = np.random.default_rng(1)
    core_row = (1 << rng.integers(0, 4, L)).astype(np.uint8)
    out = []
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, (rng.random(d.pan_size) < 0.5).astype(np.uint8))
        sim.run_generations(0, gens)
        counts = sim.core_allele_counts()
        anc = np.searchsorted(np.array([1, 2, 4, 8]), core_row)
        a = N - counts[np.arange(L), anc].astype(np.int64)
        pos = np.flatnonzero(np.minimum(a, N - a) >= 1)
        kw = -(-N // 64) * 2
        for md, bw in WINDOWS:
            site_ms, tr_ms, pair_ms, pairs = sim.ld_kernel_ms(md, bw, 1, kernel_reps)
            tiles, diag = tile_pairs(pos, md)
            work = (tiles - diag) * 128 * 128 + diag * 128 * 127 // 2
            tr_bytes = N * ((L + 15) // 16) * 4 + len(pos) * kw * 4
            ops = 2 * kw * 32 * 128 * 128 * tiles
            res = sim.core_ld(md, bw)                                   # warm-up of the end-to-end call
            assert int(res.pairs.sum()) == pairs
            times = []
            for _ in range(reps):
                t = time.perf_counter()
                sim.core_ld(md, bw)
                times.append(time.perf_counter() - t)
            med = statistics.median(times)
            out.append({
                "config": name, "pop_size": N, "core_size": L, "max_dist": md, "bin_width": bw,
                "state": f"{gens} generations from a clonal start" + ("" if core_mu is None else f" at core_mu {core_mu}"),
                "sites_used": int(res.sites_used), "pairs": pairs, "tile_pairs": tiles,
                "share_of_tile_work_in_window": pairs / work if work else None,
                "kernels": {"reps": kernel_reps, "site_pass_ms": site_ms, "transpose_ms": tr_ms, "pair_pass_ms": pair_ms,
                            "transpose_bytes": tr_bytes,
                            "transpose_gbs": tr_bytes / (tr_ms * 1e-3) / 1e9 if tr_ms else None,
                            "transpose_frac_of_hbm_copy": tr_bytes / (tr_ms * 1e-3) / 1e9 / HBM_GBS if tr_ms else None,
                            "pairs_per_s": pairs / (pair_ms * 1e-3) if pair_ms else None,
                            "i8_tensor_tops": ops / (pair_ms * 1e-3) / 1e12 if pair_ms else None,
                            "i8_frac_of_datasheet_dense": ops / (pair_ms * 1e-3) / 1e12 / INT8_TOPS_DATASHEET if pair_ms else None},
                "end_to_end": {"reps": reps, "median_ms": med * 1e3, "all_ms": [t * 1e3 for t in times],
                               "pairs_per_s": pairs / med},
                "mean_r2_first_bins": [float(x) for x in res.mean_r2[:3]],
                "four_gamete_share": float(res.four_gamete.sum()) / max(1, pairs)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--kernel_reps", type=int, default=10)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    args = ap.parse_args()
    want = args.shapes.split(",")
    res = {"gpu": gpu_info(), "hbm_gbs_reference": HBM_GBS, "int8_tops_datasheet_dense": INT8_TOPS_DATASHEET, "cases": []}
    for s in SHAPES:
        if s[0] in want:
            res["cases"] += case(*s, args.reps, args.kernel_reps)
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
