"""Clonal genealogy on the device: the record equals the parent vectors of every entry point that advances a
generation (ring wrap and resets included); the node table, its summary and the TMRCA equal a numpy trace of the
downloaded record (tests/genealogy_reference.py); hand-built histories give hand-written Newick strings; the mean
pairwise TMRCA of a neutral population matches the Wright-Fisher expectation; column shards and groups record the same
genealogy; --print_genealogy in both command lines."""
import os
import subprocess
import sys

import numpy as np
import pytest

import pansim_b200 as pb
from pansim_b200.simulate import initial_rows, sample_pairs, selection_coefficients

from genealogy_reference import NONE, np_genealogy, np_tmrca_lca, np_tmrca_walk, newick_tmrca, parse_newick

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_INVALID, ERR_STATE = -1, -5


def params(N, L=5000, selection=False, **kw):
    """selection=False: every weight equal (no selection, no genome-size control, no competition), so the parents are
    uniform draws; selection=True: the cfg2 mix of selection and competition, which coalesces fast."""
    base = dict(pop_size=N, core_size=L, pan_genes=200, core_genes=50, core_mu=1e-3, HR_rate=0.0, HGT_rate=0.05, seed=3)
    if selection:
        base.update(prop_positive=0.1, competition_strength=0.5)
    else:
        base.update(prop_positive=-0.1, no_control_genome_size=True, competition_strength=0.0)
    base.update(kw)
    return pb.Params(**base)


def started(p, **kw):
    """A context at the clonal start of p's command line (the same host draws as simulate.run)."""
    d = pb.derive(p)
    rng = np.random.default_rng(p.seed)
    sel = selection_coefficients(p, d.pan_size, rng)
    core_row, acc_row = initial_rows(p, d, rng)
    s = pb.Pansim.from_params(p, **kw)
    s.set_initial(core_row, acc_row)
    s.set_selection(sel)
    return s


def assert_reference(g, H, N):
    parent, ind, time, lin = np_genealogy(H, N)
    assert g.n_nodes == len(parent) and g.lineages_at_start == lin and g.generations_kept == len(H)
    assert (g.parent == parent).all() and (g.individual == ind).all() and (g.time == time).all()
    return parent, time


# ---- recording ---------------------------------------------------------------------------------------------------

def test_record_before_enabling_is_refused():
    with started(params(20)) as s:
        s.step(0)
        for call in (s.genealogy, s.genealogy_history, lambda: s.tmrca([0], [1])):
            with pytest.raises(pb.PansimError) as e:
                call()
            assert e.value.code == ERR_STATE
        s.enable_genealogy(4)
        s.step(1)
        assert s.genealogy_history().shape == (1, 20)
        s.enable_genealogy(0)                                          # off again
        with pytest.raises(pb.PansimError):
            s.genealogy()
        s.step(2)


def test_history_equals_the_parents_of_each_step():
    with started(params(100, selection=True)) as s:
        s.enable_genealogy(50)
        got = []
        for g in range(7):
            s.step(g)
            got.append(s.parents())
        assert (s.genealogy_history() == np.stack(got)).all()
        info = s.genealogy()
        assert (info.generations_total, info.generations_kept) == (7, 7)


@pytest.mark.parametrize("selection", [False, True])
def test_batches_record_what_single_steps_record(selection):
    p = params(300, selection=selection)
    n = 12                                                             # >= 8: the selection chain runs as graph launches
    with started(p) as a:
        a.enable_genealogy(n)
        for g in range(n):
            a.step(g)
        want = a.genealogy_history()
    r1, r2 = sample_pairs(p, np.random.default_rng(1))
    for run in (lambda s: s.run_generations(0, n), lambda s: s.run_generations_stats(0, n, r1, r2),
                lambda s: s.run_generations_diversity(0, n), lambda s: s.run_generations_diversity(0, n, r1, r2)):
        with started(p) as s:
            s.enable_genealogy(n)
            run(s)
            assert (s.genealogy_history() == want).all()


def test_ring_keeps_the_newest_vectors():
    p = params(64, selection=True)
    with started(p) as full:
        full.enable_genealogy(40)
        full.run_generations(0, 30)
        H = full.genealogy_history()
        assert H.shape == (30, 64)
    for cap in (1, 7, 29, 30, 31):
        with started(p) as s:
            s.enable_genealogy(cap)
            s.run_generations(0, 10)
            for g in range(10, 30):
                s.step(g)
            kept = min(cap, 30)
            assert (s.genealogy_history() == H[30 - kept:]).all(), cap
            g = s.genealogy()
            assert (g.generations_total, g.generations_kept) == (30, kept)
            assert_reference(g, H[30 - kept:], 64)


def test_set_initial_and_uploads_clear_the_record():
    p = params(32)
    with started(p) as s:
        s.enable_genealogy(10)
        s.run_generations(0, 3)
        core, acc = s.download_core(), s.download_acc()
        for reset in (lambda: s.set_initial(core[0], acc[0]), lambda: s.upload(core_onehot=core),
                      lambda: s.upload(acc=acc)):
            s.step(5)
            assert s.genealogy().generations_total > 0
            reset()
            g = s.genealogy()
            assert s.genealogy_history().shape == (0, 32)
            assert (g.generations_total, g.generations_kept, g.n_nodes, g.lineages_at_start) == (0, 0, 33, 32)
            assert (g.time == 0).all() and g.individual[-1] == NONE


# ---- the tree against the reference ------------------------------------------------------------------------------

TREE_CASES = [(2, 30, False), (3, 30, False), (100, 1000, False), (1000, 3000, False), (1000, 50, False),
              (100, 60, True), (1000, 100, True)]


@pytest.mark.parametrize("N,gens,selection", TREE_CASES)
def test_tree_equals_the_reference_trace(N, gens, selection):
    with started(params(N, selection=selection)) as s:
        s.enable_genealogy(gens)
        s.run_generations(0, gens)
        H = s.genealogy_history()
        g = s.genealogy()
        parent, time = assert_reference(g, H, N)
        assert g.newick() == pb.genealogy_newick(parent, g.individual, time, N)
        rng = np.random.default_rng(N)
        r1, r2 = rng.integers(0, N, 2000), rng.integers(0, N, 2000)
        r1[:5] = r2[:5]                                                 # i = j
        t = s.tmrca(r1, r2)
        assert (t == np_tmrca_lca(parent, time, r1, r2)).all() and (t == np_tmrca_walk(H, N, r1, r2)).all()
        assert (t[:5] == 0).all()
    if N == 1000 and gens == 50:
        assert g.lineages_at_start > 1 and g.individual[-1] == NONE and g.time[-1] == 50      # the virtual root
    if N == 100 and gens == 1000:
        assert g.lineages_at_start == 1 and g.time[-1] < 1000                                  # the MRCA, found early


def test_tmrca_of_all_pairs_and_a_bad_index():
    N = 200
    with started(params(N)) as s:
        s.enable_genealogy(500)
        s.run_generations(0, 500)
        H = s.genealogy_history()
        g = s.genealogy()
        parent, time = assert_reference(g, H, N)
        r1, r2 = np.triu_indices(N, 1)
        t = s.tmrca(r1, r2)
        assert (t == np_tmrca_lca(parent, time, r1, r2)).all() and (t == np_tmrca_walk(H, N, r1, r2)).all()
        for bad in (([0, N], [1, 2]), ([0, 1], [1, N + 7])):
            with pytest.raises(pb.PansimError) as e:
                s.tmrca(*bad)
            assert e.value.code == ERR_INVALID
        assert (s.tmrca(r1, r2) == t).all()                             # still usable
        s.step(500)                                                     # the record changed: traced again
        H = s.genealogy_history()
        parent, _, time, _ = np_genealogy(H, N)
        assert (s.tmrca(r1[:999], r2[:999]) == np_tmrca_lca(parent, time, r1[:999], r2[:999])).all()


# ---- hand-built histories ----------------------------------------------------------------------------------------

def test_identity_parents_never_merge():
    N = 6
    with started(params(N)) as s:
        s.enable_genealogy(8)
        for g in range(5):
            s.step_with_parents(g, np.arange(N))
        g = s.genealogy()
        assert (g.n_nodes, g.lineages_at_start) == (N + 1, N)
        assert g.newick() == "(" + ",".join(f"ind_{i}:5" for i in range(N)) + ");\n"
        assert list(s.tmrca([0, 1, 2], [5, 1, 4])) == [5, 0, 5]


def test_all_zero_parents_make_a_star():
    N = 7
    with started(params(N)) as s:
        s.enable_genealogy(8)
        s.step_replay(np.zeros(N, np.uint32))                          # H_1: everyone descends from individual 0
        s.next_generation(np.arange(N))
        s.next_generation(np.arange(N))
        g = s.genealogy()
        assert (g.n_nodes, g.lineages_at_start, g.individual[-1], g.time[-1]) == (N + 1, 1, 0, 3)
        assert g.newick() == "(" + ",".join(f"ind_{i}:3" for i in range(N)) + ");\n"


def test_designed_caterpillar():
    # going back from the present, leaf k + 1 joins the lineage of leaves 0 .. k one generation further back each time
    H = [[0, 1, 2, 3, 0], [0, 1, 2, 0, 4], [0, 1, 0, 3, 4], [0, 0, 2, 3, 4]]
    with started(params(5)) as s:
        s.enable_genealogy(4)
        s.step_with_parents(0, H[0])
        s.next_generation(H[1])
        s.step_replay(H[2])
        s.step_with_parents(3, H[3])
        g = s.genealogy()
        assert g.newick() == "((((ind_0:1,ind_1:1):1,ind_2:2):1,ind_3:3):1,ind_4:4);\n"
        assert list(g.individual[5:]) == [0, 0, 0, 0] and g.lineages_at_start == 1
        assert list(s.tmrca([0, 0, 0, 0, 3], [1, 2, 3, 4, 4])) == [1, 2, 3, 4, 4]
        s.enable_genealogy(4)                                          # enabling again clears
        assert s.genealogy().generations_total == 0


# ---- semantics ---------------------------------------------------------------------------------------------------

def test_mean_pairwise_tmrca_is_N_under_equal_weights():
    """Haploid Wright-Fisher with equal weights: two lineages meet with probability 1/N per generation, so a pair's
    TMRCA is geometric with mean N (T = 40 N: not meeting has probability e^-40). Over the N(N-1)/2 pairs of one
    population the mean shares one genealogy; its coalescent variance is N^2 * 2(n^2 + n + 3) / (9 n (n - 1)) with
    n = N (Tajima 1983, the genealogical term of Var(pi)): standard deviation 0.48 N at N = 50. R independent
    replicates (other generation numbers, so other Philox counters) give a mean with standard deviation
    0.48 N / sqrt(R); the test allows 4 of them."""
    N, T, R = 50, 2000, 40
    r1, r2 = np.triu_indices(N, 1)
    means = []
    with started(params(N, L=1000)) as s:
        s.enable_genealogy(T)
        for r in range(R):
            s.set_initial(np.full(1000, 1, np.uint8), np.zeros(s.G, np.uint8))     # a fresh start clears the record
            s.run_generations(r * T, T)
            assert s.genealogy().lineages_at_start == 1
            means.append(s.tmrca(r1, r2).mean())
    sd = N * np.sqrt(2 * (N * N + N + 3) / (9 * N * (N - 1))) / np.sqrt(R)
    assert abs(np.mean(means) - N) < 4 * sd, (np.mean(means), sd)


def test_core_diff_follows_tmrca_without_recombination():
    """With HR_rate = 0 a pair's core distance is the mutations on its two branches back to the MRCA: rank
    correlation with the TMRCA over sampled pairs (seed 3, N = 200, 400 generations, 10 SNPs per genome per
    generation). Observed on a B200: rho = 0.930. Most sampled pairs meet at one of the few deepest nodes, so the
    TMRCA takes few distinct values with many ties while core_diff varies by the Poisson spread of the mutations;
    that likely keeps rho below 1."""
    from scipy.stats import spearmanr
    p = params(200, L=100_000, core_mu=1e-4)
    r1, r2 = sample_pairs(pb.Params(pop_size=200, max_distances=3000), np.random.default_rng(7))
    with started(p) as s:
        s.enable_genealogy(400)
        s.run_generations(0, 400)
        cd = s.pair_counts(r1, r2)[0]
        rho = spearmanr(cd, s.tmrca(r1, r2))[0]
    print(f"spearman rho(core_diff, TMRCA) = {rho:.4f}")
    assert rho > 0.9, rho


# ---- shards ------------------------------------------------------------------------------------------------------

def test_column_shards_and_groups_record_one_genealogy():
    p = params(300, L=3 * 8192, selection=True)
    r1, r2 = np.random.default_rng(2).integers(0, 300, (2, 5000))
    with started(p) as whole:
        whole.enable_genealogy(40)
        whole.run_generations(0, 40)
        want, want_t = whole.genealogy(), whole.tmrca(r1, r2)
    for b, e in ((0, 8192), (8192, 3 * 8192)):
        with started(p, site_begin=b, site_end=e) as s:
            s.enable_genealogy(40)
            s.run_generations(0, 40)
            got = s.genealogy()
            assert all((np.asarray(x) == np.asarray(y)).all() for x, y in zip(got, want))
            assert (s.tmrca(r1, r2) == want_t).all()
    import torch
    for n_dev in (1, 2):
        if n_dev > torch.cuda.device_count():
            continue
        d = pb.derive(p)
        rng = np.random.default_rng(p.seed)
        sel = selection_coefficients(p, d.pan_size, rng)
        core_row, acc_row = initial_rows(p, d, rng)
        with pb.PansimGroup(p, n_dev) as g:
            g.set_initial(core_row, acc_row)
            g.set_selection(sel)
            g.enable_genealogy(40)
            g.run_generations(0, 40)
            got = g.genealogy()
            assert all((np.asarray(x) == np.asarray(y)).all() for x, y in zip(got, want))
            assert (g.tmrca(r1, r2) == want_t).all()
            assert g.genealogy_history().shape == (40, 300)


# ---- command lines -----------------------------------------------------------------------------------------------

CLI_COMMON = ["--pop_size", "40", "--core_size", "9192", "--pan_genes", "90", "--core_genes", "30", "--n_gen", "60",
              "--max_distances", "70", "--HR_rate", "0.5", "--core_mu", "0.01", "--seed", "9"]
WEIGHTED = ["--competition_strength", "0.3", "--prop_positive", "0.2"]
EQUAL = ["--no_control_genome_size"]
OTHER_FILES = (".tsv", "_per_gen.tsv", "_freqs.txt", "_diversity.tsv", "_core_sfs.txt", "_core_genome.csv",
               "_pangenome.csv", "_core_genome.vcf")


def _check_cli(run, tmp_path, tag, extra):
    plain, gen = str(tmp_path / f"{tag}_plain"), str(tmp_path / f"{tag}_gen")
    common = [*CLI_COMMON, *extra, "--print_dist", "--print_matrices", "--print_diversity", "--print_vcf"]
    run(*common, "--outpref", plain)
    run(*common, "--print_genealogy", "--outpref", gen)
    assert not os.path.exists(plain + "_genealogy.nwk") and not os.path.exists(plain + "_tmrca.tsv")
    for suffix in OTHER_FILES:
        assert open(plain + suffix, "rb").read() == open(gen + suffix, "rb").read(), suffix
    text = open(gen + "_genealogy.nwk").read()
    assert sorted(parse_newick(text)[2]) == list(range(40))
    tmrca = np.loadtxt(gen + "_tmrca.tsv", dtype=np.int64, ndmin=1)
    assert len(tmrca) == len(open(gen + ".tsv").read().splitlines())
    assert tmrca.max() <= 60
    if "--all_pairs" in extra:
        r1, r2 = np.triu_indices(40, 1)
        assert (tmrca == newick_tmrca(text, r1, r2)).all()
    return text, tmrca


def _python_run(*args):
    r = subprocess.run([sys.executable, "-m", "pansim_b200", *args], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def _cpp_binary():
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)
    binary = os.path.join(ROOT, "pansim_b200", "pansim")

    def run(*args):
        r = subprocess.run([binary, *args], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    return run


def reference_newick_of_cli(extra):
    """Replays the Python command line's run in process: the genealogy of the reference trace of its record."""
    a = dict(zip(CLI_COMMON[::2], CLI_COMMON[1::2]))
    p = pb.Params(pop_size=40, core_size=9192, pan_genes=90, core_genes=30, n_gen=60, max_distances=70, HR_rate=0.5,
                  core_mu=0.01, seed=int(a["--seed"]), no_control_genome_size="--no_control_genome_size" in extra,
                  competition_strength=0.3 if "--competition_strength" in extra else 0.0,
                  prop_positive=0.2 if "--prop_positive" in extra else -0.1)
    with started(p) as s:
        s.enable_genealogy(60)
        s.run_generations(0, 60)
        H = s.genealogy_history()
        rng = np.random.default_rng(p.seed)
        d = pb.derive(p)
        selection_coefficients(p, d.pan_size, rng)
        initial_rows(p, d, rng)
        r1, r2 = sample_pairs(p, rng)
    parent, ind, time, _ = np_genealogy(H, 40)
    return pb.genealogy_newick(parent, ind, time, 40), np_tmrca_lca(parent, time, r1, r2)


@pytest.mark.parametrize("weights", ["weighted", "equal"])
@pytest.mark.parametrize("all_pairs", [False, True])
def test_python_cli_print_genealogy(tmp_path, weights, all_pairs):
    extra = (WEIGHTED if weights == "weighted" else EQUAL) + (["--all_pairs"] if all_pairs else [])
    text, tmrca = _check_cli(_python_run, tmp_path, "py", extra)
    want_text, want_tmrca = reference_newick_of_cli(extra)
    assert text == want_text
    if not all_pairs:
        assert (tmrca == want_tmrca).all()


@pytest.mark.parametrize("all_pairs", [False, True])
def test_cpp_cli_print_genealogy(tmp_path, all_pairs):
    """The C++ command line; with all weights equal the parents depend only on the seed, so both command lines write
    the same genealogy byte for byte (their host RNGs differ, which changes the rows and the pairs, not the parents).
    --gpus 2 equals --gpus 1 where two GPUs exist."""
    run = _cpp_binary()
    extra = EQUAL + (["--all_pairs"] if all_pairs else [])
    text, _ = _check_cli(run, tmp_path, "cpp", extra)
    _check_cli(run, tmp_path, "cppw", WEIGHTED + (["--all_pairs"] if all_pairs else []))
    assert text == reference_newick_of_cli(extra)[0]
    import torch
    if torch.cuda.device_count() >= 2:
        assert _check_cli(run, tmp_path, "cpp2", extra + ["--gpus", "2"])[0] == text
