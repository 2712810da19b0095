"""Parsimony on the true genealogy on the device: core_parsimony and gene_parsimony equal the numpy reference
(tests/parsimony_reference.py) on the downloaded states and the traced genealogy (summary, per-character scores and
per-branch arrays), on evolved states of several shapes, on uploaded alignments over random trees with large
polytomies, with forced scratch slabs, on a hand-built history, through refusals, on groups of 2 and 3 shards, and in
both command lines with --print_parsimony."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import pansim_b200 as pb
from pansim_b200.simulate import initial_rows, selection_coefficients

import parsimony_reference as ref

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


def same_float(a, b):
    return (math.isnan(a) and math.isnan(b)) or a == b


def check_against_reference(s, parent):
    """Every output of both calls equals the reference on the downloaded state; returns the two results."""
    parent = np.asarray(parent, np.uint32)
    codes = CODE[s.download_core()]
    pres = s.download_acc()
    cp, gp = s.core_parsimony(parent), s.gene_parsimony(parent)
    want_sum, want_sites, want_branch = ref.core_parsimony(parent, codes)
    assert tuple(cp[:6]) == want_sum
    assert (cp.site_changes == want_sites).all() and (cp.branch_changes == want_branch).all()
    ci, ri = ref.indices(want_sum)
    assert same_float(cp.ci, ci) and same_float(cp.ri, ri)
    want_sum, want_genes, gains, losses = ref.gene_parsimony(parent, pres)
    assert tuple(gp[:6]) == want_sum
    assert (gp.gene_changes == want_genes).all() and (gp.gains == gains).all() and (gp.losses == losses).all()
    ci, ri = ref.indices(want_sum)
    assert same_float(gp.ci, ci) and same_float(gp.ri, ri)
    # the reconstruction is optimal: its changes add up to the tree length
    assert int(cp.branch_changes.sum()) == cp.tree_length and cp.branch_changes[-1] == 0
    assert int(gp.gains.sum() + gp.losses.sum()) == gp.tree_length and gp.gains[-1] == gp.losses[-1] == 0
    return cp, gp


# ---- evolved states on the traced genealogy ------------------------------------------------------------------

@pytest.mark.parametrize("shape", ["equal_weights_virtual_root", "cfg2_mrca", "hr_on", "n1", "n2"])
def test_device_equals_reference_on_evolved_states(shape):
    p, n_gen = {
        "equal_weights_virtual_root": (params(300), 6),
        "cfg2_mrca": (params(200, selection=True), 80),
        "hr_on": (params(150, HR_rate=0.5), 30),
        "n1": (params(1, HGT_rate=0.0), 5),
        "n2": (params(2), 7),
    }[shape]
    assert p.core_size % 32 and p.core_size > 8192
    with started(p) as s:
        assert s.G % 32, s.G
        s.enable_genealogy(n_gen)
        s.run_generations(0, n_gen)
        g = s.genealogy()
        if shape == "equal_weights_virtual_root":
            assert g.lineages_at_start > 40 and g.individual[-1] == NONE      # the root is a large polytomy
        if shape == "cfg2_mrca":
            assert g.lineages_at_start == 1
        cp, gp = check_against_reference(s, g.parent)
        # the defaults take the genealogy themselves
        d = s.core_parsimony()
        assert tuple(d[:8]) == tuple(cp[:8]) or all(same_float(a, b) for a, b in zip(d[:8], cp[:8]))
        assert (d.site_changes == cp.site_changes).all()
        if shape not in ("n1", "n2"):
            assert cp.variable > 0 and gp.variable > 0


# ---- uploaded alignments on random trees -----------------------------------------------------------------------

@pytest.mark.parametrize("seed", [1, 2, 3])
def test_uploaded_alignments_on_trees_with_large_polytomies(seed):
    rng = np.random.default_rng(seed)
    N = 130
    p = params(N, L=8192 + 8192 // 2 + 5)
    with pb.Pansim.from_params(p) as s:
        core = (1 << rng.integers(0, 4, (N, p.core_size))).astype(np.uint8)
        # a few columns of low diversity so that sets intersect
        core[:, :500] = np.where(rng.random((N, 500)) < 0.9, 1, core[:, :500]).astype(np.uint8)
        acc = (rng.random((N, s.G)) < rng.random(s.G)).astype(np.uint8)
        s.upload(core, acc)
        trees = [ref.random_tree(rng, N, max_children=60), ref.random_tree(rng, N, max_children=2),
                 np.array([N] * N + [NONE], np.uint32)]                          # the star: one polytomy of N
        for t in trees:
            assert max(np.bincount(t[:-1].astype(np.int64))) >= 2
            check_against_reference(s, t)
        assert max(np.bincount(trees[0][:-1].astype(np.int64))) >= 40


def test_forced_slabs_give_identical_bytes(monkeypatch):
    with started(params(300)) as s:
        s.enable_genealogy(12)
        s.run_generations(0, 12)
        g = s.genealogy()
        base = (s.core_parsimony(g), s.gene_parsimony(g))
        _, _, slabs = s.parsimony_kernel_ms(g, repeats=1)
        monkeypatch.setenv("PANSIM_PARSIMONY_SCRATCH_MB", "1")
        small = (s.core_parsimony(g), s.gene_parsimony(g))
        _, _, many = s.parsimony_kernel_ms(g, repeats=1)
        _, _, many_genes = s.parsimony_kernel_ms(g, genes=True, repeats=1)
        assert slabs == 1 and many >= 3 and many_genes >= 1
        for a, b in zip(base, small):
            for x, y in zip(a, b):
                if isinstance(x, np.ndarray):
                    assert x.tobytes() == y.tobytes()
                else:
                    assert same_float(x, y) if isinstance(x, float) else x == y
        check_against_reference(s, g.parent)


# ---- a hand-built history ------------------------------------------------------------------------------------------

def test_hand_built_history_two_independent_mutations():
    N, site = 4, 9000
    p = params(N, HGT_rate=0.0)
    d = pb.derive(p)
    with pb.Pansim.from_params(p) as s:
        core_row = np.ones(p.core_size, np.uint8)                            # all A
        s.set_initial(core_row, np.zeros(d.pan_size, np.uint8))
        s.enable_genealogy(4)
        s.step_replay(np.array([0, 0, 2, 2], np.uint32))                     # ((0, 1), (2, 3)) below generation 0
        s.step_replay(np.arange(N, dtype=np.uint32),
                      core_mut=(np.array([0, 2], np.uint32), np.array([site, site], np.uint32), np.array([2, 2], np.uint8)))
        g = s.genealogy()
        assert g.n_nodes == 7 and list(g.parent) == [4, 4, 5, 5, 6, 6, NONE]
        cp = s.core_parsimony(g)
        want = np.zeros(p.core_size, np.uint32)
        want[site] = 2
        assert (cp.site_changes == want).all()
        assert cp.branch_changes.tolist() == [1, 0, 1, 0, 0, 0, 0]
        assert tuple(cp[:6]) == (p.core_size, 1, 2, 1, 2, 1)
        assert cp.ci == 0.5 and cp.ri == 0.0
        gp = s.gene_parsimony(g)
        assert gp.tree_length == 0 and math.isnan(gp.ci) and math.isnan(gp.ri)


# ---- refusals ------------------------------------------------------------------------------------------------------

def test_bad_tables_are_refused_and_the_context_keeps_working():
    p = params(5)
    with started(p) as s:
        s.enable_genealogy(10)
        s.run_generations(0, 10)
        g = s.genealogy()
        good = check_against_reference(s, g.parent)
        bad = [np.array([5, 5, 5, 5, 5], np.uint32),                         # no root last
               np.array([5, 5, 5, 5, NONE], np.uint32)[:4],                  # fewer nodes than leaves
               np.array([5, 5, 6, 6, 7, 7, 8, 8, 9, NONE], np.uint32),       # more than 2N - 1 nodes
               np.array([3, 5, 5, 6, 6, 6, NONE], np.uint32),                # a leaf as parent
               np.array([5, 5, 6, 6, 6, 4, NONE], np.uint32),                # a parent below its child
               np.array([5, 5, 6, 6, 9, 6, NONE], np.uint32),                # a parent out of range
               np.array([6, 6, 5, 6, 6, 6, NONE], np.uint32)]                # an internal node with one child
        for t in bad:
            with pytest.raises(pb.PansimError) as e:
                s.core_parsimony(t)
            assert e.value.code == ERR_INVALID
            with pytest.raises(pb.PansimError) as e:
                s.gene_parsimony(t)
            assert e.value.code == ERR_INVALID
        again = check_against_reference(s, g.parent)
        assert (again[0].site_changes == good[0].site_changes).all()
        s.run_generations(10, 2)                                            # still steps
    with pb.Pansim.from_params(p) as fresh:
        for call in (fresh.core_parsimony, fresh.gene_parsimony):
            with pytest.raises(pb.PansimError) as e:
                call(np.array([5] * 5 + [NONE], np.uint32))
            assert e.value.code == ERR_STATE


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
        s.enable_genealogy(6)
        s.run_generations(0, 6)
        want = check_against_reference(s, s.genealogy().parent)
    with pb.PansimGroup(p, n_dev) as grp:
        grp.set_initial(core_row, acc_row)
        grp.set_selection(sel)
        grp.enable_genealogy(6)
        grp.run_generations(0, 6)
        got = (grp.core_parsimony(), grp.gene_parsimony())
    for a, b in zip(got, want):
        for x, y in zip(a, b):
            if isinstance(x, np.ndarray):
                assert x.tobytes() == y.tobytes()
            else:
                assert same_float(x, y) if isinstance(x, float) else x == y


# ---- both command lines ----------------------------------------------------------------------------------------

CLI_COMMON = ["--pop_size", "50", "--core_size", "9300", "--pan_genes", "300", "--core_genes", "20", "--n_gen", "40",
              "--max_distances", "40", "--HGT_rate", "0.3", "--HR_rate", "0.2", "--rate_genes1", "0.01",
              "--prop_positive", "-0.1", "--no_control_genome_size", "--competition_strength", "0.0", "--seed", "4"]
OTHER_FILES = (".tsv", "_per_gen.tsv", "_freqs.txt", "_core_genome.csv", "_pangenome.csv")
PARSIMONY_FILES = ("_parsimony.tsv", "_core_site_changes.txt", "_gene_changes.txt", "_branch_changes.tsv")


def _check_cli(run, tmp_path, tag, extra=()):
    plain, ps = str(tmp_path / f"{tag}_plain"), str(tmp_path / f"{tag}_ps")
    common = [*CLI_COMMON, *extra, "--print_dist", "--print_matrices"]
    run(*common, "--outpref", plain)
    run(*common, "--print_parsimony", "--outpref", ps)
    assert not os.path.exists(plain + "_parsimony.tsv") and not os.path.exists(ps + "_genealogy.nwk")
    for suffix in OTHER_FILES:
        assert open(plain + suffix, "rb").read() == open(ps + suffix, "rb").read(), suffix
    lines = open(ps + "_parsimony.tsv").read().splitlines()
    assert [ln.split("\t")[0] for ln in lines] == ["core", "genes"]
    core, genes = ([int(x) for x in ln.split("\t")[1:7]] for ln in lines)
    sites = np.loadtxt(ps + "_core_site_changes.txt", dtype=np.int64)
    gene_sc = np.loadtxt(ps + "_gene_changes.txt", dtype=np.int64)
    branch = np.loadtxt(ps + "_branch_changes.tsv", dtype=np.int64, ndmin=2)
    assert core[0] == 9300 == len(sites) and core[2] == sites.sum() == branch[:, 5].sum()
    assert genes[0] == len(gene_sc) and genes[2] == gene_sc.sum() == branch[:, 6].sum() + branch[:, 7].sum()
    assert core[2] > 0 and genes[2] > 0
    # the states of the matrices give the same scores as the reference on the branch table's tree
    n_nodes = len(branch) + 1
    parent = np.full(n_nodes, NONE, np.uint32)
    parent[branch[:, 0]] = branch[:, 1]
    codes = np.array([[{"A": 0, "C": 1, "G": 2, "T": 3}[c] for c in ln.split(",")] for ln in
                      open(ps + "_core_genome.csv").read().splitlines()], np.uint8)
    assert (ref.core_parsimony(parent, codes)[1] == sites).all()
    pres = np.array([ln.split(",")[20:] for ln in open(ps + "_pangenome.csv").read().splitlines()], np.int64)
    want = ref.gene_parsimony(parent, pres)
    assert (want[1] == gene_sc).all() and (want[2][:-1] == branch[:, 6]).all() and (want[3][:-1] == branch[:, 7]).all()
    tree = b"".join(b"\t".join(ln.split(b"\t")[:5]) + b"\n" for ln in open(ps + "_branch_changes.tsv", "rb").read().splitlines())
    return tree, b"".join(open(ps + f, "rb").read() for f in PARSIMONY_FILES)


def test_both_command_lines_print_parsimony(tmp_path):
    def run_py(*args):
        r = subprocess.run([sys.executable, "-m", "pansim_b200", *args], cwd=ROOT, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    binary = os.path.join(ROOT, "pansim_b200", "pansim")
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)

    def run_cpp(*args):
        r = subprocess.run([binary, *args], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    # Under equal weights the parents depend only on the seed, so both command lines trace the same genealogy and
    # write the same tree columns; their host RNGs draw different starting rows, so the counts are each checked
    # against the reference on the host's own matrices instead.
    py = _check_cli(run_py, tmp_path, "py")
    cpp = _check_cli(run_cpp, tmp_path, "cpp")
    assert py[0] == cpp[0]
    if _n_gpus() >= 2:
        assert _check_cli(run_cpp, tmp_path, "cpp2", extra=("--gpus", "2")) == cpp
