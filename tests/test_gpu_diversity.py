"""Core-genome diversity on the device: integer parity with numpy on download_core(), the exact identity
sum over sites == sum over all pairs of core_diff, batch == one generation at a time, shards, and the
--print_diversity outputs of both command lines."""
import os
import subprocess
import sys

import numpy as np
import pytest

import pansim_b200 as pb
from helpers import sample_pairs

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CODES = np.array([1, 2, 4, 8], np.uint8)


def np_counts(core):
    return np.stack([(core == v).sum(axis=0) for v in CODES], axis=1).astype(np.uint32)


def np_diversity(core, anc=None):
    N, L = core.shape
    n = np_counts(core).astype(np.int64)
    present = (n > 0).sum(axis=1)
    pd = int(((N * N - (n * n).sum(axis=1)) // 2).sum())
    d = pb.Diversity(L, int((present >= 2).sum()), int((present >= 3).sum()), pd)
    if anc is None:
        return d, None
    k = N - n[np.arange(L), np.searchsorted(CODES, anc)]
    return d, np.bincount(k, minlength=N + 1).astype(np.uint64)


def _sim(N, L, **kw):
    return pb.Pansim.from_params(pb.Params(pop_size=N, core_size=L, pan_genes=40, core_genes=10, HR_rate=0.0,
                                           HGT_rate=0.0, **kw))


SHAPES = [(3, 9), (7, 8191), (4, 8193), (2, 70001), (1, 17), (5, 16), (33, 1024 * 3 + 1), (130, 8192 * 2 + 5), (300, 2049)]


@pytest.mark.parametrize("N,L", SHAPES)
def test_counts_and_summaries_match_numpy(N, L):
    rng = np.random.default_rng(N * 100003 + L)
    anc = (1 << rng.integers(0, 4, L)).astype(np.uint8)
    with _sim(N, L) as sim:
        sim.set_initial(anc, np.zeros(30, np.uint8))
        d, sfs = sim.core_diversity(sfs=True)
        assert d == pb.Diversity(L, 0, 0, 0)
        assert sfs[0] == L and sfs[1:].sum() == 0
        # random state with a few columns fixed (non-segregating) and some with exactly 2 / 3 alleles
        core = (1 << rng.integers(0, 4, (N, L))).astype(np.uint8)
        core[:, ::5] = anc[::5]
        core[:, 1::7] = np.where(rng.random((N, len(range(1, L, 7)))) < 0.5, 1, 4)
        sim.upload(core)
        assert (sim.download_core() == core).all()
        assert (sim.core_allele_counts() == np_counts(core)).all()
        want, want_sfs = np_diversity(core, anc)
        assert sim.core_diversity() == want
        got, got_sfs = sim.core_diversity(sfs=True)
        assert got == want
        assert got_sfs.dtype == np.uint64 and (got_sfs == want_sfs).all()


def test_sfs_needs_set_initial():
    N, L = 6, 300
    rng = np.random.default_rng(4)
    with _sim(N, L) as sim:
        core = (1 << rng.integers(0, 4, (N, L))).astype(np.uint8)
        sim.upload(core, np.zeros((N, 30), np.uint8))
        assert sim.core_diversity() == np_diversity(core)[0]
        with pytest.raises(pb.PansimError) as e:
            sim.core_diversity(sfs=True)
        assert e.value.code == -5


def _evolved(N, L, n_gen, seed=3):
    p = pb.Params(pop_size=N, core_size=L, pan_genes=300, core_genes=100, n_gen=n_gen, HR_rate=0.5, core_mu=0.02,
                  prop_positive=0.1, competition_strength=0.4, seed=seed)
    d = pb.derive(p)
    rng = np.random.default_rng(seed)
    core_row = (1 << rng.integers(0, 4, L)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < 0.3).astype(np.uint8)
    sel = rng.normal(0, 0.05, d.pan_size)
    return p, core_row, acc_row, sel


@pytest.mark.parametrize("N,L,n_gen", [(200, 8192 * 9 + 77, 6), (1000, 1_200_000, 3)])
def test_pair_diff_sum_equals_all_pairs_core_diff(N, L, n_gen):
    p, core_row, acc_row, sel = _evolved(N, L, n_gen)
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(sel)
        for g in range(n_gen):
            sim.step(g)                 # recombination stays deferred until a reader materialises it
        d = sim.core_diversity()
        total = 0
        for _, _, cd, _, _ in sim.iter_all_pairs(chunk_pairs=4_000_000, with_indices=False):
            total += int(cd.astype(np.uint64).sum())
        assert d.pair_diff_sum == total
        assert d.segregating > 0
        if N <= 200:
            core = sim.download_core()
            want, want_sfs = np_diversity(core, core_row)
            got, got_sfs = sim.core_diversity(sfs=True)
            assert got == want and (got_sfs == want_sfs).all()


def test_batch_equals_generation_by_generation():
    N, L, n = 120, 8192 * 3 + 501, 11
    p, core_row, acc_row, sel = _evolved(N, L, n, seed=7)
    rng = np.random.default_rng(8)
    r1, r2 = sample_pairs(rng, N, 2000)

    def fresh():
        s = pb.Pansim.from_params(p)
        s.set_initial(core_row, acc_row)
        s.set_selection(sel)
        return s

    with fresh() as a:
        step_divs = []
        for g in range(n):
            a.step(g)
            step_divs.append(a.core_diversity())
        step_state = (a.download_core(), a.download_acc())
    with fresh() as b:
        divs, st = b.run_generations_diversity(0, n)
        assert st is None
        assert divs == step_divs
        assert (b.download_core() == step_state[0]).all() and (b.download_acc() == step_state[1]).all()
    with fresh() as c:
        c.run_generations(0, n)
        assert (c.download_core() == step_state[0]).all() and (c.download_acc() == step_state[1]).all()
    with fresh() as e:
        want_stats = e.run_generations_stats(0, n, r1, r2)
        want_state = (e.download_core(), e.download_acc())
    with fresh() as f:
        divs, st = f.run_generations_diversity(0, n, r1, r2)
        assert divs == step_divs
        assert st.tobytes() == want_stats.tobytes()
        assert (f.download_core() == want_state[0]).all() and (f.download_acc() == want_state[1]).all()
        # a second batch continues from the state the first left
        more, _ = f.run_generations_diversity(n, 3)
        g_last = f.core_diversity()
        assert more[-1] == g_last


def _group_case(n_dev):
    p = pb.Params(pop_size=96, core_size=8192 * 7 + 123, pan_genes=700, core_genes=200, n_gen=4, max_distances=500,
                  seed=5, prop_positive=0.1, competition_strength=0.3, HR_rate=0.5)
    d = pb.derive(p)
    rng = np.random.default_rng(1)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < 0.25).astype(np.uint8)
    sel = rng.normal(0, 0.05, d.pan_size)
    r1, r2 = sample_pairs(rng, p.pop_size, p.max_distances)
    with pb.Pansim.from_params(p) as whole:
        whole.set_initial(core_row, acc_row)
        whole.set_selection(sel)
        wdivs, wst = whole.run_generations_diversity(0, p.n_gen, r1, r2)
        wd, wsfs = whole.core_diversity(sfs=True)
        wcounts = whole.core_allele_counts()
    with pb.PansimGroup(p, n_dev) as g:
        g.set_initial(core_row, acc_row)
        g.set_selection(sel)
        divs, st = g.run_generations_diversity(0, p.n_gen, r1, r2)
        assert divs == wdivs and st.tobytes() == wst.tobytes()
        gd, gsfs = g.core_diversity(sfs=True)
        assert gd == wd and (gsfs == wsfs).all()
        assert (g.core_allele_counts() == wcounts).all()
        more, none = g.run_generations_diversity(p.n_gen, 2)
        assert none is None and more[-1] == g.core_diversity()


def test_group_one_device_matches_single_context():
    _group_case(1)


def test_group_two_devices_matches_single_context():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _group_case(2)


CLI_COMMON = ["--pop_size", "40", "--core_size", "8300", "--pan_genes", "90", "--core_genes", "30", "--n_gen", "5",
              "--max_distances", "60", "--HR_rate", "0.5", "--core_mu", "0.01", "--competition_strength", "0.3",
              "--prop_positive", "0.2", "--seed", "9"]


def _check_cli_outputs(run, tmp_path, tag):
    base, div, verb, mats = (str(tmp_path / f"{tag}_{k}") for k in ("base", "div", "verb", "mats"))
    run(*CLI_COMMON, "--print_dist", "--outpref", base)
    run(*CLI_COMMON, "--print_dist", "--print_diversity", "--outpref", div)
    run(*CLI_COMMON, "--print_diversity", "--verbose", "--outpref", verb)
    run(*CLI_COMMON, "--print_diversity", "--print_matrices", "--outpref", mats)
    for suffix in (".tsv", "_per_gen.tsv", "_freqs.txt"):
        assert open(base + suffix, "rb").read() == open(div + suffix, "rb").read(), suffix
    lines = open(div + "_diversity.tsv").read().splitlines()
    assert len(lines) == 5 and all(len(x.split("\t")) == 5 for x in lines)
    assert open(verb + "_diversity.tsv", "rb").read() == open(div + "_diversity.tsv", "rb").read()
    assert open(mats + "_diversity.tsv", "rb").read() == open(div + "_diversity.tsv", "rb").read()
    sfs = [int(x) for x in open(div + "_core_sfs.txt").read().splitlines()]
    assert len(sfs) == 41 and sum(sfs) == 8300
    assert open(verb + "_core_sfs.txt", "rb").read() == open(div + "_core_sfs.txt", "rb").read()
    # the last line from numpy over _core_genome.csv of the same run
    letters = np.array([l.split(",") for l in open(mats + "_core_genome.csv").read().splitlines()])
    core = CODES[np.searchsorted(np.array(list("ACGT")), letters)]
    d, _ = np_diversity(core)
    pi, tw, td = pb.diversity_stats(d, 40)
    assert lines[-1] == "\t".join([str(d.segregating), str(d.multiallelic), pb.fmt_f64(pi), pb.fmt_f64(tw), pb.fmt_f64(td)])
    return base, div


def test_python_cli_print_diversity(tmp_path):
    def run(*args):
        r = subprocess.run([sys.executable, "-m", "pansim_b200", *args], cwd=ROOT, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    _check_cli_outputs(run, tmp_path, "py")


def test_cpp_cli_print_diversity(tmp_path):
    binary = os.path.join(ROOT, "pansim_b200", "pansim")
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)

    def run(*args):
        r = subprocess.run([binary, *args], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    base, div = _check_cli_outputs(run, tmp_path, "cpp")
    import torch
    if torch.cuda.device_count() >= 2:
        two = str(tmp_path / "cpp_two")
        run(*CLI_COMMON, "--print_dist", "--print_diversity", "--gpus", "2", "--outpref", two)
        for suffix in (".tsv", "_per_gen.tsv", "_freqs.txt", "_diversity.tsv", "_core_sfs.txt"):
            assert open(two + suffix, "rb").read() == open(div + suffix, "rb").read(), suffix
