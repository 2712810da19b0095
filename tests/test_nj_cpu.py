"""Neighbour-joining without a device: the numpy reference (tests/nj_reference.py) recovers the generating tree of
additive metrics, pansim_tree_newick and pansim_tree_compare_splits equal the Python references on random trees with
polytomies and virtual roots (with refusals, N = 1, 2, 3 and a 100 000-leaf caterpillar), the --print_nj flag of both
command lines, and the kernels' lack of spills and stack."""
import os
import re
import subprocess

import numpy as np
import pytest

import nj_reference as ref
import parsimony_reference as pref
from pansim_b200 import NJTree, PansimError, _ffi, compare_splits, tree_newick

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CSRC = os.path.join(ROOT, "pansim_b200", "csrc")
NONE = ref.NONE
SYMBOLS = ("pansim_nj_tree", "pansim_nj_tree_matrix", "pansim_nj_kernel_ms", "pansim_tree_newick",
           "pansim_tree_compare_splits", "pansim_group_nj_tree")


def virtual_root_tree(rng, N, m):
    """A genealogy-like table: random merges until m lineages are left, then one root polytomy over them."""
    live = list(range(N))
    parent = [NONE] * N
    while len(live) > m:
        pick = rng.choice(len(live), int(rng.integers(2, min(3, len(live) - m + 1) + 1)), replace=False)
        for i in sorted(pick.tolist(), reverse=True):
            parent[live.pop(i)] = len(parent)
        live.append(len(parent))
        parent.append(NONE)
    for i in live:
        parent[i] = len(parent)
    parent.append(NONE)
    return np.array(parent, np.uint32)


@pytest.mark.parametrize("seed", range(8))
def test_reference_recovers_additive_trees(seed):
    rng = np.random.default_rng(seed)
    for N, cat in ((4, False), (9, False), (23, True), (40, False), (31, True)):
        parent, length = ref.random_binary_tree(rng, N, caterpillar=cat)
        D = ref.tree_metric(parent, length, N)
        p, l = ref.nj(D)
        assert len(p) == 2 * N - 2 and p[-1] == NONE and l[-1] == 0
        sa, sb, sh = ref.compare_splits(p, parent, N)
        assert sa == sb == sh == N - 3
        pref.validate(p, N)
        # the branch lengths of an additive metric come back too (up to rounding), through the unrooted tree
        D2 = ref.tree_metric(p, l, N)
        assert np.allclose(D2, D, atol=1e-9)


def test_reference_small_n():
    p, l = ref.nj(np.zeros((1, 1)))
    assert p.tolist() == [NONE] and l.tolist() == [0.0]
    p, l = ref.nj(np.array([[0.0, 3.0], [3.0, 0.0]]))
    assert p.tolist() == [2, 2, NONE] and l.tolist() == [1.5, 1.5, 0.0]
    D = np.array([[0, 3, 4], [3, 0, 5], [4, 5, 0]], np.float64)
    p, l = ref.nj(D)
    assert p.tolist() == [3, 3, 3, NONE] and l.tolist() == [1.0, 2.0, 3.0, 0.0]


def test_reference_ties_choose_the_first_pair():
    # every pair equidistant: every Q ties, so slots 0 and 1 join first, then the new node (slot 0) and slot 1 again
    N = 6
    D = np.ones((N, N)) - np.eye(N)
    p, _ = ref.nj(D)
    assert p[0] == p[1] == N and p[N] == p[2] == N + 1


@pytest.mark.parametrize("seed", range(10))
def test_compare_splits_equals_leaf_sets(seed):
    rng = np.random.default_rng(seed)
    for _ in range(6):
        N = int(rng.integers(2, 40))
        trees = [pref.random_tree(rng, N, max_children=int(rng.integers(2, 7))), ref.random_binary_tree(rng, N)[0],
                 np.array([N] * N + [NONE], np.uint32)]
        if N >= 6:
            trees.append(virtual_root_tree(rng, N, int(rng.integers(3, 6))))
        for a in trees:
            for b in trees:
                got = compare_splits(a, b, N)
                want = ref.compare_splits(a, b, N)
                assert (got.splits_a, got.splits_b, got.shared) == want
                assert got.rf == want[0] + want[1] - 2 * want[2]


def test_compare_splits_binary_root_counts_once():
    # ((0,1),(2,3)): the two root edges cut the same bipartition
    parent = np.array([4, 4, 5, 5, 6, 6, NONE], np.uint32)
    assert compare_splits(parent, parent, 4) == (1, 1, 1, 0)
    star = np.array([4, 4, 4, 4, NONE], np.uint32)
    assert compare_splits(parent, star, 4) == (1, 0, 0, 1)


@pytest.mark.parametrize("n", [1, 2, 3])
def test_small_trees(n):
    parent = np.array({1: [NONE], 2: [2, 2, NONE], 3: [3, 3, 3, NONE]}[n], np.uint32)
    length = np.arange(len(parent), dtype=np.float64) * 0.25
    length[-1] = 0
    assert compare_splits(parent, parent, n) == (0, 0, 0, 0)
    assert tree_newick(parent, length, n) == ref.newick(parent, length, n)
    if n == 1:
        assert tree_newick(parent, length, 1) == "ind_0;\n"
    if n == 3:
        assert tree_newick(parent, length, 3) == "(ind_0:0,ind_1:0.25,ind_2:0.5);\n"


@pytest.mark.parametrize("seed", range(6))
def test_newick_equals_reference(seed):
    rng = np.random.default_rng(seed)
    for _ in range(5):
        N = int(rng.integers(3, 60))
        for parent in (pref.random_tree(rng, N, max_children=5), ref.random_binary_tree(rng, N)[0]):
            length = rng.normal(0, 1, len(parent)) * 10.0 ** rng.integers(-20, 20, len(parent))
            length[-1] = 0
            text = tree_newick(parent, length, N)
            assert text == ref.newick(parent, length, N)
            # the lengths round-trip
            got = [float(x) for x in re.findall(r":([^,);]+)", text)]
            assert sorted(got) == sorted(length[:-1].tolist())
            assert NJTree(parent, length, N).newick() == text


def test_refusals():
    good = np.array([4, 4, 5, 5, 6, 6, NONE], np.uint32)
    bad = [np.array([4, 4, 5, 5, 6, 6, 0], np.uint32),             # root not last
           np.array([4, 4, 5, 5, 5, 6, NONE], np.uint32),          # node 4 with one child
           np.array([1, 4, 5, 5, 6, 6, NONE], np.uint32),          # a leaf as a parent
           np.array([5, 4, 5, 5, 6, 6, NONE], np.uint32)[:6],      # too few nodes for the shape
           np.array([4, 4, 5, 5, 6, 3, NONE], np.uint32)]          # a parent below its child
    L = np.zeros(7)
    for b in bad:
        with pytest.raises(PansimError):
            compare_splits(good, b, 4)
        with pytest.raises(PansimError):
            compare_splits(b, good, 4)
        with pytest.raises(PansimError):
            tree_newick(b, L[:len(b)], 4)
    with pytest.raises(PansimError):
        compare_splits(good, good, 5)
    with pytest.raises(PansimError):
        compare_splits(good, good, 0)
    assert _ffi.lib().pansim_tree_compare_splits(good.ctypes.data, 7, good.ctypes.data, 7, 4, None) == -1


def test_caterpillar_of_100000_leaves():
    N = 100_000
    # ((((0,1),2),3)...): node N joins leaves 0 and 1, node N + t joins node N + t - 1 and leaf t + 1
    parent = np.empty(2 * N - 1, np.uint32)
    parent[0] = parent[1] = N
    parent[2:N] = np.arange(N + 1, 2 * N - 1)
    parent[N:2 * N - 2] = np.arange(N + 1, 2 * N - 1)
    parent[-1] = NONE
    length = np.full(len(parent), 0.5)
    length[-1] = 0
    assert compare_splits(parent, parent, N) == (N - 3, N - 3, N - 3, 0)
    star = np.array([N] * N + [NONE], np.uint32)
    assert compare_splits(parent, star, N) == (N - 3, 0, 0, N - 3)
    text = tree_newick(parent, length, N)
    assert text.startswith("(" * (N - 1) + "ind_0:0.5,ind_1:0.5):0.5,ind_2:0.5)")
    assert text.endswith(",ind_99999:0.5);\n") and text.count("(") == N - 1


def test_symbols_exported_and_declared():
    header = open(os.path.join(ROOT, "include", "pansim_b200.h")).read()
    for s in SYMBOLS:
        assert s in _ffi.EXPORTED and re.search(rf"\b{s}\(", header), s


def test_print_nj_flag_in_both_command_lines():
    from pansim_b200.__main__ import build_parser
    assert vars(build_parser().parse_args([]))["print_nj"] is False
    assert vars(build_parser().parse_args(["--print_nj"]))["print_nj"] is True
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)
    r = subprocess.run([os.path.join(ROOT, "pansim_b200", "pansim"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--print_nj\n" in r.stdout


@pytest.mark.skipif(not os.path.exists(NVCC), reason="no nvcc")
def test_nj_kernels_have_no_spills_and_no_stack(tmp_path):
    src = tmp_path / "k.cu"
    src.write_text('#include "nj.cuh"\n')
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-cubin",
                        "-I", CSRC, "-o", str(tmp_path / "k.cubin"), str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    info = dict(re.findall(r"Compiling entry function '(\w+)'.*?\n.*?\n\s*(\d+ bytes stack frame, \d+ bytes spill stores, "
                           r"\d+ bytes spill loads)", r.stderr))
    nj = {k: v for k, v in info.items() if "nj_" in k}
    assert len(nj) == 8, info
    assert all(v == "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" for v in nj.values()), nj
