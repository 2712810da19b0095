"""Timing of parsimony on the true genealogy (pansim_b200/csrc/parsimony.cuh), one GPU call.

  python tools/parsimony_bench.py [--out profiles/r10_parsimony_bench.json] [--reps 3] [--kernel_reps 3]

Cases, each evolved on the device from the clonal start of the command line with genealogy recording on:
  cfg1       1 000 x 1.2 Mbp x 4 000 genes, defaults, 4 000 generations (full coalescence expected)
  cfg2       the cfg1 shape under selection + competition 0.5, 100 generations
  cfg4_core  10 000 x 5 Mbp x 18 000, defaults, 300 generations: the core pass (scratch in slabs)
  cfg4_acc   10 000 x 10 kbp x 18 000, defaults, 300 generations: the gene pass
  cfg5_acc   20 000 x 10 kbp x 4 000, defaults, 300 generations: the gene pass
For each pass (core, genes):
  - the kernel time from the library's CUDA events (pansim_parsimony_kernel_ms, every slab of one pass, mean of
    --kernel_reps after a warm-up), the slabs, and bytes_read = columns x (2 N x row bytes + (3 internal - 1) x set
    bytes) over that time (rows and scratch as the walk reads them);
  - end to end: pansim_core_parsimony / pansim_gene_parsimony with every output copied back, wall time around the call
    (it synchronises), median of --reps;
  - the numpy reference (tests/parsimony_reference.py) on the same genealogy and states: wall time, checked equal to
    the device's outputs. For the core it runs on the first --ref_sites sites (for cfg4 those of a column-shard
    context of the same run, which computes the same states and genealogy) and its time is also given scaled to every
    site (labelled as scaled).
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
from pansim_b200.simulate import initial_rows, selection_coefficients  # noqa: E402
import parsimony_reference as ref  # noqa: E402

CODE = np.zeros(256, np.uint8)
CODE[[1, 2, 4, 8]] = [0, 1, 2, 3]
CASES = [
    ("cfg1", dict(pop_size=1000, core_size=1_200_000, pan_genes=6000), 4000, ("core", "genes")),
    ("cfg2", dict(pop_size=1000, core_size=1_200_000, pan_genes=6000, prop_positive=0.1, competition_strength=0.5), 100,
     ("core", "genes")),
    ("cfg4_core", dict(pop_size=10_000, core_size=5_000_000, pan_genes=20_000), 300, ("core",)),
    ("cfg4_acc", dict(pop_size=10_000, core_size=10_000, pan_genes=20_000), 300, ("genes",)),
    ("cfg5_acc", dict(pop_size=20_000, core_size=10_000, pan_genes=6000), 300, ("genes",)),
]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def evolved(p, **kw):
    d = pb.derive(p)
    rng = np.random.default_rng(p.seed)
    sel = selection_coefficients(p, d.pan_size, rng)
    core_row, acc_row = initial_rows(p, d, rng)
    s = pb.Pansim.from_params(p, **kw)
    s.set_initial(core_row, acc_row)
    s.set_selection(sel)
    s.enable_genealogy(p.n_gen)
    s.run_generations(0, p.n_gen)
    return s


def timed(fn, reps):
    out, times = None, []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        times.append(time.perf_counter() - t0)
    return out, times


def one_pass(s, g, genes, reps, kernel_reps):
    ms, nbytes, slabs = s.parsimony_kernel_ms(g, genes=genes, repeats=kernel_reps)
    res, times = timed(lambda: (s.gene_parsimony(g) if genes else s.core_parsimony(g)), reps)
    return res, {"kernel_ms": ms, "slabs": slabs, "bytes_read": nbytes,
                 "read_gb_per_s": nbytes / (ms * 1e-3) / 1e9 if ms else None,
                 "end_to_end": {"reps": reps, "median_ms": statistics.median(times) * 1e3, "all_ms": [x * 1e3 for x in times]},
                 "summary": {f: int(getattr(res, f)) for f in pb.population.PARSIMONY_FIELDS} | {"ci": res.ci, "ri": res.ri}}


def case(name, kw, n_gen, passes, reps, kernel_reps, ref_sites):
    p = pb.Params(n_gen=n_gen, seed=1, **kw)
    t0 = time.perf_counter()
    s = evolved(p)
    g = s.genealogy()
    out = {"config": name, "params": kw, "generations": n_gen, "evolve_s": time.perf_counter() - t0,
           "genealogy": {"n_nodes": int(g.n_nodes), "lineages_at_start": int(g.lineages_at_start),
                         "max_children": int(np.bincount(g.parent[:-1].astype(np.int64)).max())}}
    if "core" in passes:
        res, out["core"] = one_pass(s, g, False, reps, kernel_reps)
        if p.core_size <= 2_000_000:
            codes = CODE[s.download_core()[:, :ref_sites]]
        else:
            # a column shard of the first ref_sites sites evolves the same columns and the same genealogy
            with evolved(p, site_begin=0, site_end=ref_sites) as sh:
                codes = CODE[sh.download_core()]
                assert (sh.genealogy().parent == g.parent).all()
        t0 = time.perf_counter()
        want = ref.core_parsimony(g.parent, codes)
        t = time.perf_counter() - t0
        assert (res.site_changes[:ref_sites] == want[1]).all()
        out["core"]["numpy_reference_sites"] = ref_sites
        out["core"]["numpy_reference_s"] = t
        out["core"]["numpy_reference_s_scaled_to_all_sites"] = t * p.core_size / ref_sites
        out["core"]["numpy_equal_to_device_on_those_sites"] = True
    if "genes" in passes:
        res, out["genes"] = one_pass(s, g, True, reps, kernel_reps)
        pres = s.download_acc()
        t0 = time.perf_counter()
        want = ref.gene_parsimony(g.parent, pres)
        out["genes"]["numpy_reference_s"] = time.perf_counter() - t0
        assert tuple(res[:6]) == want[0] and (res.gene_changes == want[1]).all()
        assert (res.gains == want[2]).all() and (res.losses == want[3]).all()
        out["genes"]["numpy_equal_to_device"] = True
    s.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kernel_reps", type=int, default=3)
    ap.add_argument("--ref_sites", type=int, default=8192, help="core: the sites the numpy reference runs on")
    ap.add_argument("--cases", default=",".join(c[0] for c in CASES))
    args = ap.parse_args()
    want = args.cases.split(",")
    res = {"gpu": gpu_info(), "cases": []}
    for c in CASES:
        if c[0] in want:
            res["cases"].append(case(*c, args.reps, args.kernel_reps, args.ref_sites))
            print(json.dumps(res["cases"][-1]), flush=True)
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
