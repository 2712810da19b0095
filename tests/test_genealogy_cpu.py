"""Clonal genealogy without a device: the symbols are exported, bound and declared with the struct layouts of the
header, both command lines accept --print_genealogy, genealogy.cuh compiles for sm_100a without spills or stack, the
Newick formatter against hand-written strings (no recursion on a 10^5-leaf caterpillar), and a hand-derived example of
the numpy reference."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from genealogy_reference import NONE, np_genealogy, np_tmrca_lca, np_tmrca_walk, newick_tmrca, parse_newick
from pansim_b200 import _ffi, genealogy_newick
from pansim_b200.population import PansimError

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SYMBOLS = ("pansim_enable_genealogy", "pansim_genealogy", "pansim_genealogy_history", "pansim_genealogy_tmrca",
           "pansim_genealogy_newick", "pansim_group_enable_genealogy", "pansim_group_genealogy",
           "pansim_group_genealogy_tmrca")


def test_genealogy_symbols_exported_declared_and_bound():
    L = C.CDLL(_ffi.build())
    header = open(os.path.join(ROOT, "include", "pansim_b200.h")).read()
    for name in SYMBOLS:
        assert hasattr(L, name) and name in _ffi.EXPORTED
        assert re.search(r"\bint\s+" + name + r"\(", header), name
        assert getattr(_ffi.lib(), name).restype is C.c_int
    assert "typedef struct { uint32_t parent, individual, time; } pansim_genealogy_node;" in header
    assert ("typedef struct { uint64_t generations_total; uint32_t generations_kept, n_nodes, lineages_at_start; } "
            "pansim_genealogy_info;") in header
    assert C.sizeof(_ffi.GenealogyNode) == 12 and _ffi.GenealogyNode.time.offset == 8
    assert C.sizeof(_ffi.GenealogyInfo) == 24 and _ffi.GenealogyInfo.lineages_at_start.offset == 16


def test_print_genealogy_flag_in_both_hosts():
    from pansim_b200.__main__ import build_parser
    assert vars(build_parser().parse_args([]))["print_genealogy"] is False
    assert vars(build_parser().parse_args(["--print_genealogy"]))["print_genealogy"] is True
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)
    r = subprocess.run([os.path.join(ROOT, "pansim_b200", "pansim"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "    --print_genealogy\n" in r.stdout


NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


@pytest.mark.skipif(not os.path.exists(NVCC), reason="no nvcc")
def test_genealogy_kernels_have_no_spills_and_no_stack(tmp_path):
    src = tmp_path / "genealogy.cu"
    src.write_text('#include "genealogy.cuh"\n')
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-cubin",
                        "-I", os.path.join(ROOT, "pansim_b200", "csrc"), "-o", str(tmp_path / "g.cubin"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    info = dict(re.findall(r"Compiling entry function '(\w+)'.*?\n.*?\n\s*(\d+ bytes stack frame, \d+ bytes spill stores, \d+ bytes spill loads)",
                           r.stderr))
    gen = {k: v for k, v in info.items() if "genealogy" in k}
    assert len(gen) == 2, r.stderr
    assert all(v == "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" for v in gen.values()), gen


def newick(parent, time, n_leaves):
    parent = np.asarray(parent, np.uint32)
    return genealogy_newick(parent, np.zeros(len(parent), np.uint32), np.asarray(time, np.uint32), n_leaves)


def test_newick_star():
    # four leaves under one root at time 5
    assert newick([4, 4, 4, 4, NONE], [0, 0, 0, 0, 5], 4) == "(ind_0:5,ind_1:5,ind_2:5,ind_3:5);\n"


def test_newick_cherry_inside_a_polytomy():
    # leaves 1 and 3 merge at time 2 (node 5); the root (time 7) has children 0, node 5, 2, 4, ordered by smallest leaf
    got = newick([6, 5, 6, 5, 6, 6, NONE], [0, 0, 0, 0, 0, 2, 7], 5)
    assert got == "(ind_0:7,(ind_1:2,ind_3:2):5,ind_2:7,ind_4:7);\n"


def test_newick_virtual_root():
    # no merge within a record of 4 generations: the virtual root (individual 0xFFFFFFFF) holds every leaf
    assert newick([3, 3, 3, NONE], [0, 0, 0, 4], 3) == "(ind_0:4,ind_1:4,ind_2:4);\n"
    # an empty record: branches of length 0
    assert newick([2, 2, NONE], [0, 0, 0], 2) == "(ind_0:0,ind_1:0);\n"


def test_newick_single_leaf():
    assert newick([NONE], [0], 1) == "ind_0;\n"


def test_newick_caterpillar_of_100000_leaves_needs_no_recursion():
    n = 100_000
    # node n + k (k = 0 .. n-2) at time k + 1 joins node n + k - 1 (leaves 0, 1 for k = 0) and leaf k + 1
    parent = np.empty(2 * n - 1, np.int64)
    parent[0] = n
    parent[1:n] = n + np.arange(n - 1)
    parent[n:2 * n - 2] = np.arange(n + 1, 2 * n - 1)
    parent[2 * n - 2] = NONE
    time = np.concatenate([np.zeros(n, np.int64), np.arange(1, n)])
    want = ("(" * (n - 1) + "ind_0:1,ind_1:1)" + "".join(f":1,ind_{k + 1}:{k + 1})" for k in range(1, n - 1)) + ";\n")
    assert newick(parent, time, n) == want


def test_newick_length_query_and_refusals():
    lib = _ffi.lib()
    table = np.array([[2, 0, 0], [2, 1, 0], [NONE, 0, 3]], np.uint32)
    p = table.ctypes.data_as(C.c_void_p)
    n = C.c_size_t(0)
    assert lib.pansim_genealogy_newick(p, 3, 2, None, 0, C.byref(n)) == 0 and n.value == len("(ind_0:3,ind_1:3);\n")
    buf = C.create_string_buffer(n.value)                     # no room for the NUL
    assert lib.pansim_genealogy_newick(p, 3, 2, buf, n.value, C.byref(n)) != 0 and n.value == 19
    bad = table.copy()
    bad[0, 0] = 1                                             # a leaf as parent
    with pytest.raises(PansimError):
        genealogy_newick(bad[:, 0], bad[:, 1], bad[:, 2], 2)
    bad = table.copy()
    bad[0, 2] = 4                                             # a negative branch (leaf above its parent)
    with pytest.raises(PansimError):
        genealogy_newick(bad[:, 0], bad[:, 1], bad[:, 2], 2)
    with pytest.raises(PansimError):                          # the root is not last
        genealogy_newick([NONE, 0, 0], [0, 1, 0], [0, 0, 3], 2)


# Hand-derived example: 4 individuals over 3 generations, H_1 .. H_3 oldest first (child -> parent).
#   H_3 = [3, 1, 3, 1]: present 0 and 2 have parent 3, present 1 and 3 have parent 1 -> two merges at generation 2,
#                       ordered by smallest leaf: node 4 (leaves 0, 2; individual 3) and node 5 (leaves 1, 3; individual 1)
#   H_2 = [0, 2, 2, 0]: the two lineages (ancestors 3 and 1) go to 0 and 2 -> no merge
#   H_1 = [1, 1, 1, 1]: both go to 1 -> the MRCA, node 6 at generation 0
# node  parent  individual  time
#  0      4        0         0
#  1      5        1         0
#  2      4        2         0
#  3      5        3         0
#  4      6        3         1
#  5      6        1         1
#  6     NONE      1         3
# Newick ((ind_0:1,ind_2:1):2,(ind_1:1,ind_3:1):2);  TMRCA (0,2) = (1,3) = 1, (0,1) = (2,3) = 3.
# Without H_1 (T = 2) the two lineages stay apart: a virtual root (node 6, individual NONE, time 2) and branches of 1.
HAND_H = [[1, 1, 1, 1], [0, 2, 2, 0], [3, 1, 3, 1]]


def test_reference_hand_derived_example():
    parent, ind, time, lin = np_genealogy(HAND_H, 4)
    assert list(parent) == [4, 5, 4, 5, 6, 6, NONE] and list(ind) == [0, 1, 2, 3, 3, 1, 1]
    assert list(time) == [0, 0, 0, 0, 1, 1, 3] and lin == 1
    text = genealogy_newick(parent, ind, time, 4)
    assert text == "((ind_0:1,ind_2:1):2,(ind_1:1,ind_3:1):2);\n"
    r1, r2 = np.array([0, 1, 0, 2, 3, 0]), np.array([2, 3, 1, 3, 0, 0])
    want = [1, 1, 3, 3, 3, 0]
    assert list(np_tmrca_lca(parent, time, r1, r2)) == want
    assert list(np_tmrca_walk(HAND_H, 4, r1, r2)) == want
    assert list(newick_tmrca(text, r1, r2)) == want
    assert sorted(parse_newick(text)[2]) == [0, 1, 2, 3]
    parent, ind, time, lin = np_genealogy(HAND_H[1:], 4)
    assert list(parent) == [4, 5, 4, 5, 6, 6, NONE] and list(ind) == [0, 1, 2, 3, 3, 1, NONE]
    assert list(time) == [0, 0, 0, 0, 1, 1, 2] and lin == 2
    assert genealogy_newick(parent, ind, time, 4) == "((ind_0:1,ind_2:1):1,(ind_1:1,ind_3:1):1);\n"
    assert list(np_tmrca_walk(HAND_H[1:], 4, r1, r2)) == [1, 1, 2, 2, 2, 0]


def test_reference_random_histories_agree_with_the_walk():
    rng = np.random.default_rng(5)
    for N, T in ((2, 3), (7, 1), (30, 12), (50, 200)):
        H = rng.integers(0, N, (T, N))
        parent, ind, time, _ = np_genealogy(H, N)
        r1, r2 = np.triu_indices(N)
        assert (np_tmrca_lca(parent, time, r1, r2) == np_tmrca_walk(H, N, r1, r2)).all()
        assert (newick_tmrca(genealogy_newick(parent, ind, time, N), r1, r2) == np_tmrca_walk(H, N, r1, r2)).all()
