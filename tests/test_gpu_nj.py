"""Neighbour-joining on the device: nj_tree and nj_tree_matrix equal the numpy reference (tests/nj_reference.py) bit
for bit (parent and length, tobytes()) on evolved states of several shapes, on a clonal start full of ties, across
several compactions, on additive metrics and on a hand-built infinite-sites alignment (where the tree is recovered
exactly), through refusals, on groups of 2 and 3 shards, and in both command lines with --print_nj."""
import os
import subprocess
import sys

import numpy as np
import pytest

import pansim_b200 as pb
from pansim_b200.simulate import initial_rows, selection_coefficients

import nj_reference as ref
import parsimony_reference as pref

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_INVALID, ERR_STATE = -1, -5
NONE = ref.NONE
CODE = np.zeros(256, np.uint8)
CODE[[1, 2, 4, 8]] = [0, 1, 2, 3]


def params(N, L=8192 * 2 + 77, selection=False, **kw):
    """selection=False: every weight equal; selection=True: the cfg2 mix of selection and competition."""
    base = dict(pop_size=N, core_size=L, pan_genes=300, core_genes=20, core_mu=2e-3, HR_rate=0.0, HGT_rate=0.2,
                rate_genes1=0.02, seed=11)
    if selection:
        base.update(prop_positive=0.1, competition_strength=0.5)
    else:
        base.update(prop_positive=-0.1, no_control_genome_size=True, competition_strength=0.0)
    base.update(kw)
    return pb.Params(**base)


def started(p, **kw):
    d = pb.derive(p)
    rng = np.random.default_rng(p.seed)
    sel = selection_coefficients(p, d.pan_size, rng)
    core_row, acc_row = initial_rows(p, d, rng)
    s = pb.Pansim.from_params(p, **kw)
    s.set_initial(core_row, acc_row)
    s.set_selection(sel)
    return s


def matrices(s, p):
    """The reference core and accessory matrices of the downloaded state."""
    return (ref.core_matrix(CODE[s.download_core()], p.core_size),
            ref.acc_matrix(s.download_acc().astype(np.uint8), p.core_genes))


def same_tree(got, want):
    parent, length = want
    assert got.parent.tobytes() == parent.tobytes()
    assert got.length.tobytes() == length.tobytes()


# ---- evolved states ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("shape", ["equal_weights", "cfg2", "hr_on", "n1", "n2", "n3", "n33"])
def test_device_equals_reference_on_evolved_states(shape):
    p, n_gen = {
        "equal_weights": (params(300), 30),
        "cfg2": (params(200, selection=True), 60),
        "hr_on": (params(150, HR_rate=0.5), 30),
        "n1": (params(1, HGT_rate=0.0), 5),
        "n2": (params(2), 7),
        "n3": (params(3), 7),
        "n33": (params(33), 20),
    }[shape]
    with started(p) as s:
        s.run_generations(0, n_gen)
        core, acc = matrices(s, p)
        for metric, D in (("core", core), ("acc", acc)):
            t = s.nj_tree(metric)
            assert t.n_leaves == p.pop_size and len(t.parent) == ref.nj_nodes(p.pop_size)
            same_tree(t, ref.nj(D))
            if p.pop_size >= 3:
                pref.validate(t.parent, p.pop_size)
            assert t.newick() == ref.newick(t.parent, t.length, p.pop_size)
        if shape == "equal_weights":
            assert len(np.unique(core)) > 20 and len(np.unique(acc)) > 20


def test_clonal_start_with_many_ties():
    p = params(160, core_mu=1e-7, HGT_rate=0.01, rate_genes1=0.001)
    with started(p) as s:
        s.run_generations(0, 2)
        core, acc = matrices(s, p)
        pairs = np.triu_indices(160, 1)
        assert len(np.unique(core[pairs])) < 50                          # 12 720 pairs, a dozen distances
        for metric, D in (("core", core), ("acc", acc)):
            same_tree(s.nj_tree(metric), ref.nj(D))


@pytest.mark.parametrize("kind", ["distinct", "ties"])
def test_several_compactions(kind, monkeypatch):
    rng = np.random.default_rng(5)
    n = 1200
    if kind == "distinct":
        D = rng.uniform(0.0, 1.0, (n, n))
    else:
        D = rng.integers(0, 6, (n, n)).astype(np.float64) / 8.0
    D = np.triu(D, 1)
    D = D + D.T
    want = ref.nj(D)
    with pb.Pansim.from_params(params(4)) as s:
        t = s.nj_tree_matrix(ref.upper(D), n)
        same_tree(t, want)
        # another compaction schedule gives the same bits
        monkeypatch.setenv("PANSIM_NJ_COMPACT", "0.8")
        same_tree(s.nj_tree_matrix(ref.upper(D), n), want)


def test_kernel_ms_counts_compactions(monkeypatch):
    p = params(1100, L=8192 + 5)
    with started(p) as s:
        s.run_generations(0, 4)
        t = s.nj_tree("core")
        monkeypatch.setenv("PANSIM_NJ_COMPACT", "0.5")
        build_ms, join_ms, scanned, compactions = s.nj_kernel_ms("core", repeats=1)
        # the schedule: compact to k when k <= 0.5 x the stored dimension while that is above 512 (1100 -> 550 -> 275)
        M, want = 1100, 0
        for k in range(1100, 3, -1):
            if M > 512 and k <= 0.5 * M:
                M = k
            want += M * (M - 1) // 2 * 8
        assert build_ms > 0 and join_ms > 0 and compactions == 2 and scanned == want
        same_tree(s.nj_tree("core"), (t.parent, t.length))


# ---- additive metrics and a hand-built alignment -------------------------------------------------------------------

@pytest.mark.parametrize("seed", [0, 1, 2])
def test_matrix_on_additive_metrics_recovers_the_tree(seed):
    rng = np.random.default_rng(seed)
    with pb.Pansim.from_params(params(4)) as s:
        for n, cat in ((5, False), (70, False), (97, True), (300, False)):
            parent, length = ref.random_binary_tree(rng, n, caterpillar=cat)
            D = ref.tree_metric(parent, length, n)
            t = s.nj_tree_matrix(ref.upper(D), n)
            same_tree(t, ref.nj(D))
            assert pb.compare_splits(t, parent, n).rf == 0


def test_infinite_sites_alignment_recovers_the_tree():
    rng = np.random.default_rng(9)
    N = 64
    parent, _ = ref.random_binary_tree(rng, N)
    p = params(N, L=8192 + 8192 // 2 + 5)
    # every non-root branch carries 1 .. 40 mutations; each mutated site changes A to C below its branch only
    below = ref.leaf_sets(parent, N)
    core = np.ones((N, p.core_size), np.uint8)
    site = 0
    for v in range(len(parent) - 1):
        for _ in range(int(rng.integers(1, 41))):
            core[sorted(below[v]), site] = 2
            site += 1
    assert site < p.core_size
    with pb.Pansim.from_params(p) as s:
        s.upload(core, np.zeros((N, s.G), np.uint8))
        t = s.nj_tree("core")
        D = ref.core_matrix(CODE[core], p.core_size)
        same_tree(t, ref.nj(D))
        assert pb.compare_splits(t, parent, N) == (N - 3, N - 3, N - 3, 0)
        # the NJ table is a node table the parsimony calls accept: every site then changes once
        cp = s.core_parsimony(t.parent)
        assert cp.tree_length == site and cp.homoplastic == 0


# ---- refusals ------------------------------------------------------------------------------------------------------

def test_refusals_leave_the_context_working():
    p = params(40)
    with pb.Pansim.from_params(p) as fresh:
        for metric in ("core", "acc"):
            with pytest.raises(pb.PansimError) as e:
                fresh.nj_tree(metric)
            assert e.value.code == ERR_STATE
    with started(p) as s:
        s.run_generations(0, 5)
        want = s.nj_tree("acc")
        D = np.ones((5, 5)) - np.eye(5)
        for bad in (np.nan, -0.5, np.inf):
            u = ref.upper(D)
            u[3] = bad
            with pytest.raises(pb.PansimError) as e:
                s.nj_tree_matrix(u, 5)
            assert e.value.code == ERR_INVALID
        same_tree(s.nj_tree("acc"), (want.parent, want.length))
        same_tree(s.nj_tree_matrix(ref.upper(D), 5), ref.nj(D))
        s.run_generations(5, 2)
        core, _ = matrices(s, p)
        same_tree(s.nj_tree("core"), ref.nj(core))
    q = params(40, L=8192 * 3)
    with started(q, site_begin=8192, site_end=8192 * 2) as shard:
        shard.run_generations(0, 3)
        with pytest.raises(pb.PansimError) as e:
            shard.nj_tree("core")
        assert e.value.code == ERR_STATE
        shard.nj_tree("acc")                                      # the accessory matrix is whole on every shard
        shard.run_generations(3, 1)


# ---- groups --------------------------------------------------------------------------------------------------------

def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("n_dev", [1, 2, 3])
def test_groups_equal_the_single_context(n_dev):
    if _n_gpus() < n_dev:
        pytest.skip(f"needs {n_dev} GPUs")
    p = params(96, L=8192 * 7 + 123, selection=True, HR_rate=0.5, n_gen=6)
    d = pb.derive(p)
    rng = np.random.default_rng(p.seed)
    sel = selection_coefficients(p, d.pan_size, rng)
    core_row, acc_row = initial_rows(p, d, rng)
    with pb.Pansim.from_params(p) as s:
        s.set_initial(core_row, acc_row)
        s.set_selection(sel)
        s.run_generations(0, 6)
        want = [s.nj_tree(m) for m in ("core", "acc")]
    with pb.PansimGroup(p, n_dev) as grp:
        grp.set_initial(core_row, acc_row)
        grp.set_selection(sel)
        grp.run_generations(0, 6)
        for m, w in zip(("core", "acc"), want):
            same_tree(grp.nj_tree(m), (w.parent, w.length))


# ---- both command lines --------------------------------------------------------------------------------------------

CLI_COMMON = ["--pop_size", "50", "--core_size", "9300", "--pan_genes", "300", "--core_genes", "20", "--n_gen", "40",
              "--max_distances", "40", "--HGT_rate", "0.3", "--HR_rate", "0.2", "--rate_genes1", "0.01",
              "--prop_positive", "-0.1", "--no_control_genome_size", "--competition_strength", "0.0", "--seed", "4"]
OTHER_FILES = (".tsv", "_per_gen.tsv", "_freqs.txt", "_core_genome.csv", "_pangenome.csv")
NJ_FILES = ("_core_nj.nwk", "_acc_nj.nwk", "_nj_rf.tsv")


def _check_cli(run, tmp_path, tag, extra=()):
    plain, nj = str(tmp_path / f"{tag}_plain"), str(tmp_path / f"{tag}_nj")
    common = [*CLI_COMMON, *extra, "--print_dist", "--print_matrices"]
    run(*common, "--outpref", plain)
    run(*common, "--print_nj", "--outpref", nj)
    assert not os.path.exists(plain + "_nj_rf.tsv") and not os.path.exists(nj + "_genealogy.nwk")
    for suffix in OTHER_FILES:
        assert open(plain + suffix, "rb").read() == open(nj + suffix, "rb").read(), suffix
    # the trees are the reference's on the written matrices
    codes = np.array([[{"A": 0, "C": 1, "G": 2, "T": 3}[c] for c in ln.split(",")] for ln in
                      open(nj + "_core_genome.csv").read().splitlines()], np.uint8)
    pres = np.array([ln.split(",")[20:] for ln in open(nj + "_pangenome.csv").read().splitlines()], np.uint8)
    trees = {"core": ref.nj(ref.core_matrix(codes, 9300)), "acc": ref.nj(ref.acc_matrix(pres, 20))}
    for m, (parent, length) in trees.items():
        assert open(f"{nj}_{m}_nj.nwk").read() == ref.newick(parent, length, 50)
    lines = [ln.split("\t") for ln in open(nj + "_nj_rf.tsv").read().splitlines()]
    assert [ln[0] for ln in lines] == ["core", "acc"]
    for ln in lines:
        a, b, shared, rf = (int(x) for x in ln[1:5])
        assert a == 47 and rf == a + b - 2 * shared and float(ln[5]) == pytest.approx(rf / (a + b))
    return [ln[2] for ln in lines], b"".join(open(nj + f, "rb").read() for f in NJ_FILES)


def test_both_command_lines_print_nj(tmp_path):
    def run_py(*args):
        r = subprocess.run([sys.executable, "-m", "pansim_b200", *args], cwd=ROOT, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    binary = os.path.join(ROOT, "pansim_b200", "pansim")
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)

    def run_cpp(*args):
        r = subprocess.run([binary, *args], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    # Under equal weights both command lines trace the same genealogy (the parents depend only on the seed), so the
    # genealogy's split counts agree; their host RNGs draw different starting rows, so each tree is checked against
    # the reference on that command line's own matrices.
    py = _check_cli(run_py, tmp_path, "py")
    cpp = _check_cli(run_cpp, tmp_path, "cpp")
    assert py[0] == cpp[0]
    if _n_gpus() >= 2:
        assert _check_cli(run_cpp, tmp_path, "cpp2", extra=("--gpus", "2")) == cpp
