"""Timing of the clonal genealogy (pansim_b200/csrc/genealogy.cuh), one GPU call.

  python tools/genealogy_bench.py [--out profiles/r06_genealogy_bench.json] [--rounds 8] [--gens 1000] [--reps 5]

- Recording cost: generations per second of the cfg2 batch (1 000 x 1.2 Mbp, 4 000 accessory genes, selection and
  competition 0.5) on two contexts of the same seed, one recording (ring of 1 000 vectors) and one not, alternated
  --rounds times; each round is one pansim_run_generations batch of --gens generations, wall time around the call (it
  synchronises).
- Trace: wall time of pansim_genealogy right after one more generation was recorded (so it traces again), median of
  --reps; the call traces on the device and copies back the node table (at most 2N x 12 bytes). Shapes: cfg2 after
  100 generations; all weights equal (uniform parents) at N = 1 000 after 100 and 10 000 generations and at
  N = 20 000 after 1 000 generations. Lineages merge fastest in the first generations, so the work is front-loaded.
- TMRCA: wall time of pansim_genealogy_tmrca for the 10^5 sampled pairs of the cfg2 command line (median of --reps)
  and for all N(N-1)/2 = 2.0 * 10^8 pairs at N = 20 000 in row blocks of 4 * 10^6 pairs (the sum over the blocks; the
  host-side index lists are made outside the timed calls). Each call copies 12 bytes per pair over PCIe.
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
from pansim_b200.simulate import initial_rows, sample_pairs, selection_coefficients  # noqa: E402

CFG2 = dict(pop_size=1000, core_size=1_200_000, pan_genes=6000, core_genes=2000, max_distances=100_000,
            prop_positive=0.1, competition_strength=0.5, seed=0)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def started(p):
    d = pb.derive(p)
    rng = np.random.default_rng(p.seed)
    sel = selection_coefficients(p, d.pan_size, rng)
    core_row, acc_row = initial_rows(p, d, rng)
    s = pb.Pansim.from_params(p)
    s.set_initial(core_row, acc_row)
    s.set_selection(sel)
    return s, rng


def equal_weights(N):
    return pb.Params(pop_size=N, core_size=8192, pan_genes=200, core_genes=50, prop_positive=-0.1,
                     no_control_genome_size=True, competition_strength=0.0, seed=1)


def timed(f):
    t0 = time.perf_counter()
    out = f()
    return (time.perf_counter() - t0) * 1e3, out


def trace_case(name, p, gens, reps):
    s, _ = started(p)                                    # left open: the caller times the TMRCA on it, then closes it
    s.enable_genealogy(gens)
    s.run_generations(0, gens)
    ms = []
    for r in range(reps + 1):
        s.step(gens + r)                                 # the record changed: the next call traces again
        t, g = timed(s.genealogy)
        ms.append(t)
    ms = ms[1:]                                          # the first call loads the module
    return {"case": name, "pop_size": p.pop_size, "generations_kept": g.generations_kept, "n_nodes": g.n_nodes,
            "lineages_at_start": g.lineages_at_start, "trace_call_ms_median": statistics.median(ms),
            "trace_call_ms": ms}, s


def all_pairs_blocks(N, chunk=4_000_000):
    i0 = 0
    while i0 < N - 1:
        i1, n = i0, 0
        while i1 < N - 1 and (n == 0 or n + (N - 1 - i1) <= chunk):
            n += N - 1 - i1
            i1 += 1
        rows = np.arange(i0, i1, dtype=np.int64)
        counts = N - 1 - rows
        ii = np.repeat(rows, counts)
        start = np.repeat(np.cumsum(counts) - counts, counts)
        jj = np.arange(len(ii), dtype=np.int64) - start + ii + 1
        yield ii.astype(np.uint32), jj.astype(np.uint32)
        i0 = i1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_genealogy_bench.json"))
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--gens", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    res = {"gpu": gpu_info()}

    # recording on / off, alternated
    p2 = pb.Params(**CFG2)
    off, _ = started(p2)
    on, rng = started(p2)
    r1, r2 = sample_pairs(p2, rng)
    on.enable_genealogy(1000)
    for s in (off, on):
        s.run_generations(0, 20)                         # warm-up: modules, graphs of every phase
    rounds = []
    gen = 20
    for _ in range(a.rounds):
        row = {}
        for name, s in (("off", off), ("on", on)):
            t, _ = timed(lambda: s.run_generations(gen, a.gens))
            row[name] = a.gens / (t / 1e3)
        gen += a.gens
        rounds.append(row)
        print(json.dumps(row), flush=True)
    res["recording_gens_per_s"] = {"gens_per_round": a.gens, "rounds": rounds,
                                   "off_median": statistics.median(r["off"] for r in rounds),
                                   "on_median": statistics.median(r["on"] for r in rounds)}
    assert (on.download_core() == off.download_core()).all(), "recording changed the simulated state"
    off.close()
    on.close()

    # trace
    res["trace"] = []
    cfg2_rec, s = trace_case("cfg2", pb.Params(**CFG2), 100, a.reps)
    res["trace"].append(cfg2_rec)
    with s:
        ms = []
        for _ in range(a.reps + 1):
            t, out = timed(lambda: s.tmrca(r1, r2))
            ms.append(t)
        res["tmrca_sampled"] = {"case": "cfg2", "pairs": len(r1), "call_ms_median": statistics.median(ms[1:]),
                                "call_ms": ms[1:], "mean_tmrca": float(out.mean())}
    print(json.dumps(res["trace"][-1]), json.dumps(res["tmrca_sampled"]), flush=True)
    for name, N, gens in (("equal_1k_100", 1000, 100), ("equal_1k_10000", 1000, 10000), ("equal_20k_1000", 20000, 1000)):
        rec, s = trace_case(name, equal_weights(N), gens, a.reps)
        res["trace"].append(rec)
        print(json.dumps(rec), flush=True)
        if N == 20000:
            with s:
                total, pairs = 0.0, 0
                for ii, jj in all_pairs_blocks(N):
                    t, _ = timed(lambda: s.tmrca(ii, jj))
                    total += t
                    pairs += len(ii)
                res["tmrca_all_pairs"] = {"case": name, "pairs": pairs, "call_ms_total": total,
                                          "pairs_per_s": pairs / (total / 1e3)}
                print(json.dumps(res["tmrca_all_pairs"]), flush=True)
        else:
            s.close()
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
