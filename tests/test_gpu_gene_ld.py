"""Accessory-gene linkage on the device: every output of pansim_gene_ld equals, exactly, a numpy reference over the
presence matrix (uploaded, crafted and evolved states, every compartment layout); repeated calls reuse their buffers;
groups equal the single context; errors leave the context working; --print_gene_ld in both command lines."""
import dataclasses
import os
import subprocess
import sys

import numpy as np
import pytest

import pansim_b200 as pb
from pansim_b200.params import fmt_f64

from gene_ld_reference import CLASSES, gene_groups, np_gene_ld

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def assert_equal(got, want):
    assert got.classes == CLASSES
    for f in ("pairs", "four_gamete", "associated", "dissociated"):
        assert [int(x) for x in getattr(got, f)] == want[f], (f, getattr(got, f), want[f])
    assert got.r2_sum == want["r2_sum"]
    assert (got.hist.astype(np.int64) == want["hist"]).all()
    assert (got.genes_used.astype(np.int64) == want["genes_used"]).all()
    for k in range(3):
        assert np.array_equal(got.mean_r2[k], pb.population.ld_mean_r2(want["pairs"][k], want["r2_sum"][k]), equal_nan=True)


def assert_same(got, want):
    """Two GeneLD results are equal field by field (NaN means equal NaN)."""
    assert got.classes == want.classes and got.r2_sum == want.r2_sum
    for f in ("pairs", "four_gamete", "associated", "dissociated", "mean_r2", "hist", "genes_used"):
        assert np.array_equal(getattr(got, f), getattr(want, f), equal_nan=f == "mean_r2"), f


def _cfg(N, G, layout):
    """A context of N rows and G accessory genes with a compartment layout: "one" (all group 0), "two" (group 1 from
    a boundary off every word and tile edge) or "custom" (a group-1 range inside the genes)."""
    p = pb.Params(pop_size=N, core_size=64, pan_genes=G + 10, core_genes=10, HR_rate=0.0, HGT_rate=0.0, prop_genes2=0.0)
    cfg = pb.make_config(p)
    if layout == "one":
        cfg.n_compartments, cfg.comp_lo[0], cfg.comp_hi[0] = 1, 0, G
    elif layout == "two":
        b = (2 * G) // 3
        b -= 1 if b and b % 32 == 0 else 0
        cfg.n_compartments = 2
        cfg.comp_lo[0], cfg.comp_hi[0], cfg.comp_lo[1], cfg.comp_hi[1] = 0, b, b, G
    else:
        cfg.n_compartments = 2
        cfg.comp_lo[0], cfg.comp_hi[0] = 0, G
        cfg.comp_lo[1], cfg.comp_hi[1] = min(G, G // 5 + 1), max(min(G, G // 5 + 1), G - G // 7)
    return cfg


def _groups(cfg, G):
    return gene_groups(G, cfg.n_compartments, list(cfg.comp_lo), list(cfg.comp_hi))


def forced_presence(rng, N, G, min_minor):
    """Random presence with genes forced to: present everywhere, absent everywhere, and the min_minor edges
    (min_minor - 1, min_minor, N - min_minor, N - min_minor + 1 rows), and a spread of frequencies."""
    pres = rng.random((N, G)) < rng.random(G)[None, :]
    pres[:, 0::11] = True
    pres[:, 1::13] = False
    for e, g0 in enumerate(range(2, 2 + 4 * 7, 7)):
        k = [min_minor - 1, min_minor, N - min_minor, N - min_minor + 1][e]
        for g in range(g0, G, 7 * 4):
            pres[:, g] = False
            if 0 < k <= N:
                pres[rng.permutation(N)[:k], g] = True
    return pres


NS = [2, 3, 63, 64, 65, 1000, 1100]
GS = [1, 31, 33, 127, 128, 129, 4000]


@pytest.mark.parametrize("G", GS)
@pytest.mark.parametrize("N", NS)
def test_uploaded_states_match_numpy(N, G):
    rng = np.random.default_rng(N * 7919 + G)
    sims = {lay: pb.Pansim(_cfg(N, G, lay)) for lay in ("one", "two", "custom")}
    try:
        for mm in sorted({1, 2, max(1, N // 2)}):
            pres = forced_presence(rng, N, G, mm)
            core = np.full((N, 64), 1, np.uint8)
            for lay, sim in sims.items():
                sim.upload(core, pres.astype(np.uint8))
                for bins in (1, 20, 1024):
                    if G == 4000 and N >= 1000 and (lay, bins) not in (("two", 20), ("custom", 1024), ("one", 1)):
                        continue                     # the reference walks 8e6 pairs per call at this size
                    got = sim.gene_ld(bins, mm)
                    assert_equal(got, np_gene_ld(pres, _groups(sim.cfg, G), bins, mm))
    finally:
        for s in sims.values():
            s.close()


def _upload(sim, pres):
    sim.upload(np.full((sim.N, sim.local_sites), 1, np.uint8), pres.astype(np.uint8))


def test_crafted_matrices():
    N, G = 64, 300
    rng = np.random.default_rng(5)
    with pb.Pansim(_cfg(N, G, "two")) as sim:
        grp = _groups(sim.cfg, G)
        # nested gene sets (dyadic row intervals: any two nested or disjoint) are a perfect phylogeny
        pres = np.zeros((N, G), bool)
        for g in range(G):
            size = N >> (int(rng.integers(0, 5)) + 1)
            k = int(rng.integers(0, N // size))
            pres[k * size:(k + 1) * size, g] = True
        _upload(sim, pres)
        got = sim.gene_ld(20)
        assert got.pairs.sum() > 0 and (got.four_gamete == 0).all()
        assert_equal(got, np_gene_ld(pres, grp, 20, 1))
        # identical genes: q = 2^32, every pair associated, all in the last bin
        col = rng.random(N) < 0.3
        same = np.repeat(col[:, None], G, axis=1)
        _upload(sim, same)
        got = sim.gene_ld(16)
        assert int(got.pairs.sum()) == G * (G - 1) // 2
        assert all(r == int(p) << 32 for r, p in zip(got.r2_sum, got.pairs)) and (got.associated == got.pairs).all()
        assert (got.hist[:, :-1] == 0).all() and (got.hist[:, -1] == got.pairs).all() and (got.mean_r2[got.pairs > 0] == 1.0).all()
        # complementary genes: r^2 = 1; the pairs of a gene with its complement are dissociated
        comp = np.where(np.arange(G)[None, :] % 2 == 0, col[:, None], ~col[:, None])
        _upload(sim, comp)
        got = sim.gene_ld(16)
        even, odd = (G + 1) // 2, G // 2
        assert int(got.dissociated.sum()) == even * odd
        assert int(got.associated.sum()) == even * (even - 1) // 2 + odd * (odd - 1) // 2
        assert all(r == int(p) << 32 for r, p in zip(got.r2_sum, got.pairs))
        assert_equal(got, np_gene_ld(comp, grp, 16, 1))
        # genes present or absent everywhere are never used
        pres = rng.random((N, G)) < 0.5
        pres[:, 5:40] = True
        pres[:, 200:260] = False
        _upload(sim, pres)
        got = sim.gene_ld()
        want = np_gene_ld(pres, grp, 20, 1)
        assert int(got.genes_used.sum()) == G - 35 - 60
        assert_equal(got, want)


EVOLVED = {
    "neutral": dict(pop_size=300, pan_genes=1300, core_genes=100, n_gen=6),
    "selection": dict(pop_size=257, pan_genes=1130, core_genes=100, n_gen=6, prop_positive=0.2, competition_strength=0.4,
                      genome_size_penalty=0.9),
    "low_flip_hgt": dict(pop_size=400, pan_genes=2100, core_genes=100, n_gen=30, rate_genes1=1e-4, rate_genes2=1e-2,
                         HGT_rate=0.5),
}


def _evolved(kind, seed=3):
    p = pb.Params(core_size=8192, HR_rate=0.0, core_mu=0.001, seed=seed, **{"HGT_rate": 0.0, **EVOLVED[kind]})
    d = pb.derive(p)
    rng = np.random.default_rng(seed)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < 0.5).astype(np.uint8)
    sel = rng.normal(0, 0.05, d.pan_size)
    return p, d, core_row, acc_row, sel


@pytest.mark.parametrize("kind", list(EVOLVED))
def test_evolved_states(kind):
    p, d, core_row, acc_row, sel = _evolved(kind)
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(sel)
        sim.run_generations(0, p.n_gen - 1)
        sim.step(p.n_gen - 1)                            # the last accessory step, then the call
        got = sim.gene_ld(20)
        pres = sim.download_acc().astype(bool)
        grp = _groups(sim.cfg, d.pan_size)
    assert got.genes_used.sum() > 0 and got.pairs.sum() > 0
    assert_equal(got, np_gene_ld(pres, grp, 20, 1))


def test_repeated_calls_reuse_buffers():
    p, d, core_row, acc_row, sel = _evolved("selection")
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(sel)
        sim.run_generations(0, p.n_gen)
        pres = sim.download_acc().astype(bool)
        grp = _groups(sim.cfg, d.pan_size)
        first = sim.gene_ld(20)
        counts = sim.gene_counts()
        for bins in (1024, 1, 7, 20):
            got = sim.gene_ld(bins)
            assert (got.pairs == first.pairs).all() and got.r2_sum == first.r2_sum
            assert (got.four_gamete == first.four_gamete).all() and (got.associated == first.associated).all()
            assert (got.hist.sum(axis=1) == got.pairs).all() and (got.genes_used == first.genes_used).all()
            assert_equal(got, np_gene_ld(pres, grp, bins, 1))
        assert (sim.gene_counts() == counts).all()        # the gene counts buffer is not shared
        assert_same(sim.gene_ld(20), first)
        g_ms, t_ms, q_ms, pairs = sim.gene_ld_kernel_ms(20, 1, 3)
        assert pairs == int(first.pairs.sum()) and g_ms > 0 and t_ms > 0 and q_ms > 0


@pytest.mark.parametrize("n_dev", [1, 2, 3])
def test_group_matches_single_context(n_dev):
    import torch
    if n_dev > torch.cuda.device_count():
        pytest.skip(f"needs {n_dev} GPUs")
    p, d, core_row, acc_row, sel = _evolved("low_flip_hgt")
    p = dataclasses.replace(p, core_size=8192 * 3)
    core_row = np.resize(core_row, p.core_size)
    with pb.Pansim.from_params(p) as whole:
        whole.set_initial(core_row, acc_row)
        whole.set_selection(sel)
        whole.run_generations(0, p.n_gen)
        want = whole.gene_ld(33, 2)
    with pb.PansimGroup(p, n_dev) as g:
        g.set_initial(core_row, acc_row)
        g.set_selection(sel)
        g.run_generations(0, p.n_gen)
        got = g.gene_ld(33, 2)
    assert_same(got, want)


def test_errors_and_the_context_still_works():
    N, G = 50, 140
    rng = np.random.default_rng(2)
    with pb.Pansim(_cfg(N, G, "two")) as sim:
        with pytest.raises(pb.PansimError) as e:
            sim.gene_ld()                                # no state
        assert e.value.code == -5
        pres = rng.random((N, G)) < 0.4
        sim.upload(acc=pres.astype(np.uint8))            # the accessory matrix alone is enough
        grp = _groups(sim.cfg, G)
        assert_equal(sim.gene_ld(), np_gene_ld(pres, grp, 20, 1))
        for args in ((0, 1), (1025, 1), (20, 0), (2 ** 32 - 1, 1)):
            with pytest.raises(pb.PansimError) as e:
                sim.gene_ld(*args)
            assert e.value.code == -1
            assert_equal(sim.gene_ld(1024, 3), np_gene_ld(pres, grp, 1024, 3))
    # G = 0 and N < 2 give zeros
    p = pb.Params(pop_size=1, core_size=64, pan_genes=40, core_genes=10)
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(np.full(64, 1, np.uint8), np.ones(30, np.uint8))
        got = sim.gene_ld()
        assert got.pairs.sum() == 0 and got.genes_used.sum() == 0 and got.hist.sum() == 0 and np.isnan(got.mean_r2).all()
    p = pb.Params(pop_size=20, core_size=64, pan_genes=10, core_genes=10)
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(np.full(64, 1, np.uint8), np.zeros(0, np.uint8))
        got = sim.gene_ld(5)
        assert got.pairs.sum() == 0 and got.hist.shape == (3, 5) and got.genes_used.sum() == 0


CLI_COMMON = ["--pop_size", "60", "--core_size", "9192", "--pan_genes", "700", "--core_genes", "30", "--n_gen", "12",
              "--max_distances", "60", "--HGT_rate", "0.3", "--rate_genes1", "0.001", "--rate_genes2", "0.05",
              "--competition_strength", "0.3", "--prop_positive", "0.2", "--seed", "9"]
OTHER_FILES = (".tsv", "_per_gen.tsv", "_freqs.txt", "_core_genome.csv", "_pangenome.csv", "_diversity.tsv")
GL_FLAGS = ["--gene_ld_bins", "12", "--gene_ld_min_minor", "2"]


def tsv_lines(r):
    """<outpref>_gene_ld.tsv as both command lines must write it for these reference results."""
    out = []
    for k, label in enumerate(CLASSES):
        mean = fmt_f64(pb.population.ld_mean_r2(r["pairs"][k], r["r2_sum"][k]))
        out.append("\t".join([label, str(r["pairs"][k]), str(r["four_gamete"][k]), str(r["associated"][k]),
                              str(r["dissociated"][k]), mean, *(str(int(x)) for x in r["hist"][k])]) + "\n")
    return "".join(out).encode()


def _check_cli(run, tmp_path, tag, extra=()):
    plain, gl = str(tmp_path / f"{tag}_plain"), str(tmp_path / f"{tag}_gl")
    common = [*CLI_COMMON, *extra, "--print_dist", "--print_matrices", "--print_diversity"]
    run(*common, "--outpref", plain)
    run(*common, "--print_gene_ld", *GL_FLAGS, "--outpref", gl)
    assert not os.path.exists(plain + "_gene_ld.tsv")
    for suffix in OTHER_FILES:
        assert open(plain + suffix, "rb").read() == open(gl + suffix, "rb").read(), suffix
    rows = [line.split(",")[30:] for line in open(gl + "_pangenome.csv").read().splitlines()]
    pres = np.array(rows, dtype=np.int64).astype(bool)
    d = pb.derive(pb.Params(pop_size=60, pan_genes=700, core_genes=30))
    grp = gene_groups(d.pan_size, len(d.comp), [c[0] for c in d.comp], [c[1] for c in d.comp])
    want = np_gene_ld(pres, grp, 12, 2)
    assert sum(want["pairs"]) > 0 and want["pairs"][1] > 0
    got = open(gl + "_gene_ld.tsv", "rb").read()
    assert got == tsv_lines(want)
    return got


def test_python_cli_print_gene_ld(tmp_path):
    def run(*args):
        r = subprocess.run([sys.executable, "-m", "pansim_b200", *args], cwd=ROOT, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    _check_cli(run, tmp_path, "py")


def test_cpp_cli_print_gene_ld(tmp_path):
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
