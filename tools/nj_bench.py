"""Timing of neighbour-joining on the device (pansim_b200/csrc/nj.cuh), one GPU call.

  python tools/nj_bench.py [--out profiles/r12_nj_bench.json] [--kernel_reps 2] [--compact 0.5,0.7,0.9]

Cases, each evolved on the device for a few generations from the clonal start of the command line (the join loop
depends only on N; the build on N and the row length):
  cfg1   1 000 x 1.2 Mbp x 4 000 genes, defaults, 200 generations
  cfg2   the cfg1 shape under selection + competition 0.5, 100 generations
  cfg4   10 000 x 5 Mbp x 18 000 genes, defaults, 20 generations
  cfg5   20 000 x 1.2 Mbp x 4 000 genes, defaults, 20 generations
For each metric (core, acc):
  - build and join-loop ms from the library's CUDA events (pansim_nj_kernel_ms, mean of --kernel_reps after a
    warm-up), bytes the scans read (the stored upper triangle of every iteration x 8 bytes) and that over the join
    time, against the HBM copy bandwidth measured here (a 4 GiB device-to-device copy timed with CUDA events; the
    scan reads, the copy reads and writes, so the copy's read + write bytes over its time are the yardstick);
  - the join loop's floor where it is bound by launches: ms per iteration;
  - end to end: Pansim.nj_tree wall time (it synchronises and copies the table back);
  - the numpy reference (tests/nj_reference.py) at N <= --ref_max: wall time, checked bit-equal to the device; at
    larger N its time is extrapolated from the largest measured case by N^3 and labelled so.
--compact re-runs the join loop of the cfg4 core case under each PANSIM_NJ_COMPACT fraction (the compaction choice).
The card name and power limit are read with `nvidia-smi --query-gpu=name,power.limit --format=csv` in the same call.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import pansim_b200 as pb  # noqa: E402
from pansim_b200.simulate import initial_rows, selection_coefficients  # noqa: E402
import nj_reference as ref  # noqa: E402

CODE = np.zeros(256, np.uint8)
CODE[[1, 2, 4, 8]] = [0, 1, 2, 3]
CASES = [
    ("cfg1", dict(pop_size=1000, core_size=1_200_000, pan_genes=6000), 200),
    ("cfg2", dict(pop_size=1000, core_size=1_200_000, pan_genes=6000, prop_positive=0.1, competition_strength=0.5), 100),
    ("cfg4", dict(pop_size=10_000, core_size=5_000_000, pan_genes=20_000), 20),
    ("cfg5", dict(pop_size=20_000, core_size=1_200_000, pan_genes=6000), 20),
]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def copy_bandwidth():
    """Device-to-device copy of 4 GiB, CUDA events, best of 5: bytes read + written per second."""
    import torch
    a = torch.empty(1 << 32, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    best = None
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    del a, b
    torch.cuda.empty_cache()
    return 2 * (1 << 32) / (best * 1e-3)


def evolved(p):
    d = pb.derive(p)
    rng = np.random.default_rng(p.seed)
    sel = selection_coefficients(p, d.pan_size, rng)
    core_row, acc_row = initial_rows(p, d, rng)
    s = pb.Pansim.from_params(p)
    s.set_initial(core_row, acc_row)
    s.set_selection(sel)
    s.run_generations(0, p.n_gen)
    return s


def metric_pass(s, p, metric, kernel_reps, hbm, ref_max, ref_time):
    N = p.pop_size
    build_ms, join_ms, scanned, compactions = s.nj_kernel_ms(metric, repeats=kernel_reps)
    t0 = time.perf_counter()
    tree = s.nj_tree(metric)
    wall = time.perf_counter() - t0
    out = {"build_ms": build_ms, "join_ms": join_ms, "iterations": max(N - 3, 0), "us_per_iteration": join_ms * 1e3 / max(N - 3, 1),
           "bytes_scanned": scanned, "scan_tb_per_s": scanned / (join_ms * 1e-3) / 1e12,
           "scan_share_of_copy_bandwidth": scanned / (join_ms * 1e-3) / hbm, "compactions": compactions,
           "end_to_end_ms": wall * 1e3}
    if N <= ref_max:
        if metric == "core":
            D = ref.core_matrix(CODE[s.download_core()], p.core_size)
        else:
            D = ref.acc_matrix(s.download_acc().astype(np.uint8), p.core_genes)
        t0 = time.perf_counter()
        parent, length = ref.nj(D)
        t = time.perf_counter() - t0
        assert parent.tobytes() == tree.parent.tobytes() and length.tobytes() == tree.length.tobytes()
        out["numpy_reference_s"] = t
        out["numpy_equal_to_device"] = True
        ref_time[metric] = (N, t)
    elif metric in ref_time:
        n0, t0 = ref_time[metric]
        out["numpy_reference_s_extrapolated_by_N3"] = t0 * (N / n0) ** 3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--kernel_reps", type=int, default=2)
    ap.add_argument("--ref_max", type=int, default=1000)
    ap.add_argument("--compact", default="0.5,0.7,0.8,0.9,0.95")
    ap.add_argument("--cases", default=",".join(c[0] for c in CASES))
    args = ap.parse_args()
    want = args.cases.split(",")
    res = {"gpu": gpu_info(), "hbm_copy_bytes_per_s": copy_bandwidth(), "cases": []}
    ref_time = {}
    for name, kw, n_gen in CASES:
        if name not in want:
            continue
        p = pb.Params(n_gen=n_gen, seed=1, **kw)
        t0 = time.perf_counter()
        s = evolved(p)
        out = {"config": name, "params": kw, "generations": n_gen, "evolve_s": time.perf_counter() - t0}
        for metric in ("core", "acc"):
            out[metric] = metric_pass(s, p, metric, args.kernel_reps, res["hbm_copy_bytes_per_s"], args.ref_max, ref_time)
        if name == "cfg4" and args.compact:
            out["compaction_fraction"] = {}
            for f in args.compact.split(","):
                os.environ["PANSIM_NJ_COMPACT"] = f
                b, j, nb, nc = s.nj_kernel_ms("core", repeats=1)
                out["compaction_fraction"][f] = {"join_ms": j, "bytes_scanned": nb, "compactions": nc}
            os.environ.pop("PANSIM_NJ_COMPACT", None)
        s.close()
        res["cases"].append(out)
        print(json.dumps(out), flush=True)
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
