"""Core-genome LD on the device: every bin field and the used-site count equal, exactly, a numpy reference over
download_core() and the ancestral row; perfect phylogenies have no four-gamete pair; the deferred recombination is
materialised first; shard contexts chained through `next` and groups sum to the single context; errors; --print_ld in
both command lines."""
import ctypes as C
import dataclasses
import os
import subprocess
import sys

import numpy as np
import pytest

import pansim_b200 as pb
from pansim_b200.params import fmt_f64

from ld_reference import np_ld_from_derived

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CODES = np.array([1, 2, 4, 8], np.uint8)


def np_ld(core, anc, max_dist, bin_width, min_minor=1, site_begin=0):
    return np_ld_from_derived(core != anc[None, :], max_dist, bin_width, min_minor, site_begin)


def assert_equal(got, want):
    pairs, fg, r2, used = want
    assert got.sites_used == used
    assert (got.pairs.astype(np.int64) == pairs).all(), (got.pairs, pairs)
    assert (got.four_gamete.astype(np.int64) == fg).all()
    assert got.r2_sum == r2
    for k in range(len(pairs)):
        assert np.array_equal(got.mean_r2[k], pb.population.ld_mean_r2(int(pairs[k]), r2[k]), equal_nan=True)


def _sim(N, L, **kw):
    return pb.Pansim.from_params(pb.Params(pop_size=N, core_size=L, pan_genes=40, core_genes=10, HR_rate=0.0,
                                           HGT_rate=0.0, **kw))


def forced_state(rng, N, L, anc, min_minor):
    """Random rows with columns forced to: every row ancestral, fixed derived, singletons, the min_minor edges
    (min_minor - 1, min_minor, N - min_minor, N - min_minor + 1 derived rows) and 3 or 4 letters."""
    core = (1 << rng.integers(0, 4, (N, L))).astype(np.uint8)
    code = np.searchsorted(CODES, anc)

    def other(s, k=0):
        return CODES[(code[s] + 1 + k) % 4]

    for s in range(0, L, 11):
        core[:, s] = anc[s]                                          # every row ancestral
    for s in range(1, L, 13):
        core[:, s] = other(s)                                        # fixed derived
    for s in range(2, L, 17):
        core[:, s] = anc[s]
        core[rng.integers(0, N), s] = other(s, int(rng.integers(0, 3)))   # singleton
    for e, s0 in enumerate(range(3, 3 + 4 * 19, 19)):
        k = [min_minor - 1, min_minor, N - min_minor, N - min_minor + 1][e]
        for s in range(s0, L, 19 * 4):
            core[:, s] = anc[s]
            if 0 < k <= N:
                core[rng.permutation(N)[:k], s] = other(s, int(rng.integers(0, 3)))
    for s in range(5, L, 23):                                        # multiallelic
        core[:, s] = CODES[rng.integers(0, 4, N)]
    return core


SHAPES = [(3, 9), (7, 8191), (4, 8193), (2, 70001), (1, 17), (5, 16), (33, 1024 * 3 + 1), (130, 8192 * 2 + 5),
          (300, 2049), (600, 70001), (1100, 5003)]
WINDOWS = [(1, 1), (100, 7), (300, 1000), ("L", "L")]


@pytest.mark.parametrize("N,L", SHAPES)
def test_bins_match_numpy(N, L):
    rng = np.random.default_rng(N * 7919 + L)
    anc = (1 << rng.integers(0, 4, L)).astype(np.uint8)
    with _sim(N, L) as sim:
        sim.set_initial(anc, np.zeros(30, np.uint8))
        clonal = sim.core_ld(100, 7)
        assert clonal.sites_used == 0 and (clonal.pairs == 0).all() and np.isnan(clonal.mean_r2).all()
        for min_minor in (1, 2):
            core = forced_state(rng, N, L, anc, min_minor)
            sim.upload(core)
            for md, bw in WINDOWS:
                if md == "L":
                    if L > 10000:
                        continue                     # the numpy reference would walk 1e8 to 2.4e9 pairs
                    md = bw = L
                got = sim.core_ld(md, bw, min_minor)
                assert_equal(got, np_ld(core, anc, md, bw, min_minor))
                assert (got.dist_lo == np.arange(len(got.pairs)) * bw + 1).all()
                assert got.dist_hi[-1] == md


def nested_clades(N, L, rng):
    """Derived sets that are dyadic row intervals: any two are nested or disjoint, a perfect phylogeny."""
    der = np.zeros((N, L), bool)
    for s in range(L):
        lev = int(rng.integers(0, int(np.log2(N))))
        size = N >> (lev + 1)
        k = int(rng.integers(0, N // size))
        der[k * size:(k + 1) * size, s] = True
    return der


def derived_to_core(der, anc):
    code = np.searchsorted(CODES, anc)
    return np.where(der, CODES[(code + 1) % 4][None, :], anc[None, :]).astype(np.uint8)


def test_perfect_phylogeny_recombinant_and_identical_columns():
    N, L = 64, 3000
    rng = np.random.default_rng(5)
    anc = (1 << rng.integers(0, 4, L)).astype(np.uint8)
    der = nested_clades(N, L, rng)
    with _sim(N, L) as sim:
        sim.set_initial(anc, np.zeros(30, np.uint8))
        sim.upload(derived_to_core(der, anc))
        got = sim.core_ld(L, 50)
        assert got.pairs.sum() > 0 and (got.four_gamete == 0).all()
        assert_equal(got, np_ld_from_derived(der, L, 50, 1))
        # one recombinant row: row 0 carries row N - 1's alleles at the first half of the sites and its own at the
        # second; a pair (s, t) across the breakpoint with row N - 1's clade at s and row 0's clade at t now shows
        # all four gametes. The brute force below counts the four-gamete pairs directly.
        rec = der.copy()
        rec[0, :L // 2] = der[N - 1, :L // 2]
        sim.upload(derived_to_core(rec, anc))
        got = sim.core_ld(L, 50)
        g = rec.astype(np.int64)
        four = 0
        for s in range(0, L):
            t = np.arange(s + 1, L)
            both = g[:, s:s + 1] & g[:, t]
            c = both.sum(0)
            a_s, a_t = g[:, s].sum(), g[:, t].sum(0)
            ok = (min(a_s, N - a_s) >= 1) & (np.minimum(a_t, N - a_t) >= 1)
            four += int((ok & (c > 0) & (a_s - c > 0) & (a_t - c > 0) & (N - a_s - a_t + c > 0)).sum())
        assert int(got.four_gamete.sum()) == four > 0
        assert_equal(got, np_ld_from_derived(rec, L, 50, 1))
        # identical columns: r^2 = 1, q = 2^32 for every pair
        same = np.repeat(der[:, :1], L, axis=1)
        sim.upload(derived_to_core(same, anc))
        got = sim.core_ld(1000, 100)
        assert got.pairs.sum() > 0
        assert all(r == int(p) << 32 for r, p in zip(got.r2_sum, got.pairs)) and (got.four_gamete == 0).all()


def test_evolved_state_is_materialised_first():
    p = pb.Params(pop_size=150, core_size=8192 * 4 + 999, pan_genes=300, core_genes=100, n_gen=4, HR_rate=0.5,
                  core_mu=0.01, prop_positive=0.1, competition_strength=0.4, seed=11)
    d = pb.derive(p)
    rng = np.random.default_rng(11)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < 0.3).astype(np.uint8)
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(rng.normal(0, 0.05, d.pan_size))
        for g in range(p.n_gen):
            sim.step(g)                                 # recombination stays deferred
        got = sim.core_ld(2000, 100)                    # LD first: it must materialise
        core = sim.download_core()
    assert got.sites_used > 1000
    assert_equal(got, np_ld(core, core_row, 2000, 100))


def _shard_case():
    p = pb.Params(pop_size=90, core_size=8192 * 3 + 500, pan_genes=300, core_genes=100, n_gen=4, HR_rate=0.5,
                  core_mu=0.02, seed=6, prop_positive=0.1, competition_strength=0.3)
    d = pb.derive(p)
    rng = np.random.default_rng(6)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < 0.25).astype(np.uint8)
    sel = rng.normal(0, 0.05, d.pan_size)
    return p, core_row, acc_row, sel


def _bounds(L, n, i):
    b, e = C.c_uint64(), C.c_uint64()
    assert pb._ffi.lib().pansim_shard_bounds(L, n, i, C.byref(b), C.byref(e)) == 0
    return b.value, e.value


def _sum(parts):
    return (sum(x.sites_used for x in parts), sum(x.pairs.astype(np.int64) for x in parts),
            sum(x.four_gamete.astype(np.int64) for x in parts), [sum(r) for r in zip(*(x.r2_sum for x in parts))])


WIN_SHARDS = [(300, 7), (500, 50), (1, 1)]


@pytest.mark.parametrize("n_shards", [2, 3])
def test_shards_chained_through_next_sum_to_the_whole(n_shards):
    p, core_row, acc_row, sel = _shard_case()
    with pb.Pansim.from_params(p) as whole:
        whole.set_initial(core_row, acc_row)
        whole.set_selection(sel)
        whole.run_generations(0, p.n_gen)
        want = [whole.core_ld(md, bw) for md, bw in WIN_SHARDS]
        core = whole.download_core()
    for (md, bw), w in zip(WIN_SHARDS, want):
        assert_equal(w, np_ld(core, core_row, md, bw))
    shards = []
    try:
        for i in range(n_shards):
            b, e = _bounds(p.core_size, n_shards, i)
            s = pb.Pansim.from_params(p, site_begin=b, site_end=e)
            shards.append(s)
            s.set_initial(core_row, acc_row)
            s.set_selection(sel)
            s.run_generations(0, p.n_gen)
        for (md, bw), w in zip(WIN_SHARDS, want):
            parts = [s.core_ld(md, bw, next=shards[i + 1] if i + 1 < n_shards else None) for i, s in enumerate(shards)]
            used, pairs, fg, r2 = _sum(parts)
            assert used == w.sites_used and (pairs == w.pairs.astype(np.int64)).all()
            assert (fg == w.four_gamete.astype(np.int64)).all() and r2 == w.r2_sum
            alone = [s.core_ld(md, bw) for s in shards]              # without next: only the pairs inside each shard
            assert _sum(alone)[1].sum() < pairs.sum() or md == 1
    finally:
        for s in shards:
            s.close()


@pytest.mark.parametrize("n_dev", [1, 2])
def test_group_matches_single_context(n_dev):
    import torch
    if n_dev > torch.cuda.device_count():
        pytest.skip("needs two GPUs")
    p, core_row, acc_row, sel = _shard_case()
    with pb.Pansim.from_params(p) as whole:
        whole.set_initial(core_row, acc_row)
        whole.set_selection(sel)
        whole.run_generations(0, p.n_gen)
        want = [whole.core_ld(md, bw) for md, bw in WIN_SHARDS]
    with pb.PansimGroup(p, n_dev) as g:
        g.set_initial(core_row, acc_row)
        g.set_selection(sel)
        g.run_generations(0, p.n_gen)
        for (md, bw), w in zip(WIN_SHARDS, want):
            got = g.core_ld(md, bw)
            assert got.sites_used == w.sites_used and (got.pairs == w.pairs).all()
            assert (got.four_gamete == w.four_gamete).all() and got.r2_sum == w.r2_sum
        with pytest.raises(pb.PansimError) as e:
            g.core_ld(p.core_size + 1, 100)              # wider than the narrowest shard
        assert e.value.code == -1


def test_errors_and_the_context_still_works():
    N, L = 6, 300
    rng = np.random.default_rng(2)
    with _sim(N, L) as sim:
        with pytest.raises(pb.PansimError) as e:
            sim.core_ld(10, 1)                           # no state
        assert e.value.code == -5
        core = (1 << rng.integers(0, 4, (N, L))).astype(np.uint8)
        sim.upload(core, np.zeros((N, 30), np.uint8))
        with pytest.raises(pb.PansimError) as e:
            sim.core_ld(10, 1)                           # uploads give no ancestral row
        assert e.value.code == -5
        sim.set_initial(core[0], np.zeros(30, np.uint8))
        sim.upload(core)
        for args in ((0, 1, 1), (10, 0, 1), (10, 1, 0)):
            with pytest.raises(pb.PansimError) as e:
                sim.core_ld(*args)
            assert e.value.code == -1
        assert_equal(sim.core_ld(50, 5), np_ld(core, core[0], 50, 5))
    p, core_row, acc_row, _ = _shard_case()
    b0, e0 = _bounds(p.core_size, 3, 0)
    b1, e1 = _bounds(p.core_size, 3, 1)
    b2, e2 = _bounds(p.core_size, 3, 2)
    q = dataclasses.replace(p, pop_size=p.pop_size + 1)
    with pb.Pansim.from_params(p, site_begin=b0, site_end=e0) as s0, \
            pb.Pansim.from_params(p, site_begin=b1, site_end=e1) as s1, \
            pb.Pansim.from_params(p, site_begin=b2, site_end=e2) as s2, \
            pb.Pansim.from_params(q, site_begin=b1, site_end=e1) as other_n:
        for s, sim_p in ((s0, p), (s1, p), (s2, p), (other_n, q)):
            d = pb.derive(sim_p)
            s.set_initial(core_row, np.zeros(d.pan_size, np.uint8))
        for nxt, md in ((s2, 10), (other_n, 10), (s1, e1 - b1 + 1), (s0, 10)):
            with pytest.raises(pb.PansimError) as e:
                s0.core_ld(md, 1, next=nxt)              # not adjacent, another N, wider than next, itself
            assert e.value.code == -1
        assert s1.core_ld(500, 50, next=s2).sites_used == 0     # clonal; the contexts still work
        assert s0.core_ld(10, 1, next=s1).sites_used == 0


CLI_COMMON = ["--pop_size", "40", "--core_size", "9192", "--pan_genes", "90", "--core_genes", "30", "--n_gen", "5",
              "--max_distances", "60", "--HR_rate", "0.5", "--core_mu", "0.01", "--competition_strength", "0.3",
              "--prop_positive", "0.2", "--seed", "9"]
OTHER_FILES = (".tsv", "_per_gen.tsv", "_freqs.txt", "_diversity.tsv", "_core_sfs.txt", "_core_genome.csv",
               "_pangenome.csv", "_core_genome.vcf")
LD_FLAGS = ["--ld_max_dist", "700", "--ld_bin_width", "30", "--ld_min_minor", "2"]


def derived_from_vcf(text, N, L):
    """derived [N, L] from a VCF body: GT != 0 <=> derived; sites without a line are ancestral in every row."""
    body = text[text.index(b"\n#CHROM"):].split(b"\n", 2)[2]
    der = np.zeros((N, L), bool)
    for line in body.splitlines():
        f = line.split(b"\t")
        der[:, int(f[1]) - 1] = np.array([g != b"0" for g in f[9:]])
    return der


def tsv_lines(ld_ref, md, bw):
    """<outpref>_core_ld.tsv as both command lines must write it for these bins."""
    pairs, fg, r2, _ = ld_ref
    out = []
    for b in range(len(pairs)):
        lo, hi = b * bw + 1, min((b + 1) * bw, md)
        out.append(f"{lo}\t{hi}\t{pairs[b]}\t{fg[b]}\t{fmt_f64(pb.population.ld_mean_r2(int(pairs[b]), r2[b]))}\n")
    return "".join(out).encode()


def _check_cli(run, tmp_path, tag, extra=()):
    plain, ld = str(tmp_path / f"{tag}_plain"), str(tmp_path / f"{tag}_ld")
    common = [*CLI_COMMON, *extra, "--print_dist", "--print_matrices", "--print_diversity", "--print_vcf"]
    run(*common, "--outpref", plain)
    run(*common, "--print_ld", *LD_FLAGS, "--outpref", ld)
    assert not os.path.exists(plain + "_core_ld.tsv")
    for suffix in OTHER_FILES:
        assert open(plain + suffix, "rb").read() == open(ld + suffix, "rb").read(), suffix
    der = derived_from_vcf(open(ld + "_core_genome.vcf", "rb").read(), 40, 9192)
    want = np_ld_from_derived(der, 700, 30, 2)
    assert want[0].sum() > 0
    got = open(ld + "_core_ld.tsv", "rb").read()
    assert got == tsv_lines(want, 700, 30)
    return got


def test_python_cli_print_ld(tmp_path):
    def run(*args):
        r = subprocess.run([sys.executable, "-m", "pansim_b200", *args], cwd=ROOT, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    _check_cli(run, tmp_path, "py")


def test_cpp_cli_print_ld(tmp_path):
    """The C++ file equals the same Python formatter applied to the reference bins (so the two hosts format bins
    byte-identically; their runs differ because their host RNGs do); --gpus 2 equals --gpus 1 where two GPUs exist."""
    binary = os.path.join(ROOT, "pansim_b200", "pansim")
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)

    def run(*args):
        r = subprocess.run([binary, *args], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    one = _check_cli(run, tmp_path, "cpp")
    import torch
    if torch.cuda.device_count() >= 2:
        two = _check_cli(run, tmp_path, "cpp2", extra=("--gpus", "2"))
        assert two == one
