"""Timing of the pangenome accumulation curves (pansim_b200/csrc/pangenome.cuh), one GPU call.

  python tools/gene_accumulation_bench.py [--out profiles/r09_gene_accumulation_bench.json] [--perms 100] [--reps 5]
                                          [--kernel_reps 10]

Shapes, each evolved on the device from a clonal start (every row the same random accessory row, so every gene
starts fixed), at the low flip rates --rate_genes1 1e-4 --rate_genes2 1e-2 with --HGT_rate 0.05, and at the default
rates (1 and 1 000 hits per gene compartment and generation):
  cfg1        1 000 x G 4 000
  cfg4_acc   10 000 x G 18 000 (a 10 kbp core: only the accessory matrix is read)
  cfg5_acc   20 000 x G 4 000
For each, at --perms orders:
  - kernel times from the library's CUDA events (pansim_gene_accumulation_kernel_ms), mean of --kernel_reps after a
    warm-up: the order draw, and the accumulation (zeroed counts, chunk summaries, walk, curves);
  - the L2-read rate bytes_read / accumulation time, bytes_read = perms * N * ceil(G / 32) * 4 (the rows as the walk
    reads them; the matrix fits in L2 at these shapes, so this is not a share of HBM bandwidth);
  - the grid: word slices x row chunks x orders, as the library plans it from the SM count;
  - end to end: pansim_gene_accumulation with every output copied back, wall time around the call (it synchronises),
    median of --reps;
  - the numpy reference (tests/gene_accumulation_reference.py) on the same orders, what a user does today from
    _pangenome.csv: wall time of its first --ref_orders orders, checked equal to the device's, and that time scaled to
    every order (labelled as scaled);
  - what the state shows: pan at k = 2, N / 2 and N (mean over orders), the spectrum's classes.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

import pansim_b200 as pb  # noqa: E402
from gene_accumulation_reference import np_curves, np_orders  # noqa: E402

LOW = dict(rate_genes1=1e-4, rate_genes2=1e-2, HGT_rate=0.05)
SHAPES = [("cfg1", 1000, 6000, 2000, 300, LOW), ("cfg4_acc", 10_000, 20_000, 2000, 100, LOW),
          ("cfg5_acc", 20_000, 6000, 2000, 100, LOW), ("cfg1_default_rates", 1000, 6000, 2000, 50, {}),
          ("cfg4_acc_default_rates", 10_000, 20_000, 2000, 50, {}), ("cfg5_acc_default_rates", 20_000, 6000, 2000, 50, {})]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


WALK_CTAS_PER_SM = 6    # pg_walk_kernel: 74 registers x 128 threads (ptxas, DESIGN.md section 16)


def plan(words, N, P, sms):
    """The library's grid (pansim_b200.cu, gene_acc_plan): word slices of 128, row chunks (at most one wave of
    resident walk CTAs), orders."""
    slices = -(-words // 128)
    base = slices * P
    slots = WALK_CTAS_PER_SM * sms
    chunks = max(1, min(slots // base, N // 256)) if base < slots else 1
    rows = -(-(-(-N // chunks)) // 32) * 32
    chunks = -(-N // rows)
    return {"word_slices": slices, "row_chunks": chunks, "orders": P, "walk_ctas": slices * chunks * P,
            "walk_ctas_per_sm": slices * chunks * P / sms, "walk_waves": slices * chunks * P / slots,
            "summary_ctas": slices * (chunks - 1) * P}


def case(name, N, pan_genes, core_genes, gens, rates, perms, reps, kernel_reps, ref_orders):
    p = pb.Params(pop_size=N, core_size=10_000, pan_genes=pan_genes, core_genes=core_genes, seed=1, **rates)
    d = pb.derive(p)
    rng = np.random.default_rng(1)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, (rng.random(d.pan_size) < 0.5).astype(np.uint8))
        sim.run_generations(0, gens)
        order_ms, accum_ms, nbytes = sim.gene_accumulation_kernel_ms(perms, 7, kernel_reps)
        res = sim.gene_accumulation(perms, 7)                       # warm-up of the end-to-end call
        times = []
        for _ in range(reps):
            t = time.perf_counter()
            sim.gene_accumulation(perms, 7)
            times.append(time.perf_counter() - t)
        spec = sim.gene_spectrum()
        pres = sim.download_acc().astype(bool)
        sms = sim.info().sm_count
    # the numpy reference on the same orders: the draw, then the curves of the first ref_orders orders
    t = time.perf_counter()
    orders = np_orders(7, perms, N)
    ref_draw_s = time.perf_counter() - t
    k = min(perms, ref_orders)
    t = time.perf_counter()
    ref = np_curves(pres, orders[:k], core_genes)
    ref_curves_s = time.perf_counter() - t
    assert np.array_equal(orders, res.orders)
    assert all(np.array_equal(r, g[:k]) for r, g in zip(ref, (res.pan, res.core, res.new, res.unique)))
    med = statistics.median(times)
    classes = pb.pangenome_classes(spec, N)
    return {
        "config": name, "pop_size": N, "genes": d.pan_size, "core_genes": core_genes, "rates": rates,
        "state": f"{gens} generations from a clonal start", "perms": perms,
        "grid": plan(-(-d.pan_size // 32), N, perms, sms), "sm_count": sms,
        "kernels": {"reps": kernel_reps, "order_draw_ms": order_ms, "accumulation_ms": accum_ms, "bytes_read": nbytes,
                    "l2_read_gb_per_s": nbytes / (accum_ms * 1e-3) / 1e9 if accum_ms else None},
        "end_to_end": {"reps": reps, "median_ms": med * 1e3, "all_ms": [x * 1e3 for x in times]},
        "numpy_reference": {"order_draw_s": ref_draw_s, "curves_orders_timed": k, "curves_s": ref_curves_s,
                            "curves_s_scaled_to_all_orders": ref_curves_s * perms / k, "equal_to_device": True},
        "state_summary": {"pan_mean_at_k": {str(kk): float(res.pan[:, kk - 1].mean()) for kk in (1, 2, max(1, N // 2), N)},
                          "core_mean_at_N": float(res.core[:, -1].mean()),
                          "classes": dict(zip(pb.population.PANGENOME_CLASSES, classes)),
                          "spectrum_bins_1_to_5": [int(x) for x in spec[1:6]],
                          "spectrum_bins_N_minus_4_to_N": [int(x) for x in spec[-5:]]}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--perms", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--kernel_reps", type=int, default=10)
    ap.add_argument("--ref_orders", type=int, default=5, help="orders the numpy reference's curves are timed on")
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    args = ap.parse_args()
    want = args.shapes.split(",")
    res = {"gpu": gpu_info(), "cases": []}
    for s in SHAPES:
        if s[0] in want:
            res["cases"].append(case(*s, args.perms, args.reps, args.kernel_reps, args.ref_orders))
            print(json.dumps(res["cases"][-1]), flush=True)
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
