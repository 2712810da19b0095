"""Parsimony without a device: the numpy reference (tests/parsimony_reference.py) against brute-force enumeration of
every internal assignment and hand-worked trees, its table checks, pansim_parsimony_indices against the reference
(NaN cases included), the exported and declared symbols, the --print_parsimony flag of both command lines, and the
kernels' lack of spills and stack."""
import ctypes as C
import itertools
import math
import os
import re
import subprocess

import numpy as np
import pytest

import parsimony_reference as ref
from pansim_b200 import _ffi, parsimony_indices
from pansim_b200.population import PARSIMONY_FIELDS
from pansim_b200.simulate import clades

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CSRC = os.path.join(ROOT, "pansim_b200", "csrc")
NONE = ref.NONE
SYMBOLS = ("pansim_core_parsimony", "pansim_gene_parsimony", "pansim_parsimony_kernel_ms", "pansim_group_core_parsimony",
           "pansim_group_gene_parsimony")


def brute_force(parent, leaf_states, n_states):
    """The least number of branches whose ends differ, over every assignment of states to the internal nodes."""
    parent = np.asarray(parent, np.int64)
    N = leaf_states.shape[0]
    n = len(parent)
    best = np.full(leaf_states.shape[1], np.iinfo(np.int64).max)
    for assign in itertools.product(range(n_states), repeat=n - N):
        st = np.concatenate([leaf_states, np.repeat(np.array(assign, np.int64)[:, None], leaf_states.shape[1], axis=1)])
        cost = sum((st[k] != st[parent[k]]).astype(np.int64) for k in range(n - 1))
        best = np.minimum(best, cost)
    return best


@pytest.mark.parametrize("seed", range(12))
def test_reference_equals_brute_force_on_random_trees(seed):
    rng = np.random.default_rng(seed)
    for _ in range(4):
        N = int(rng.integers(2, 9))
        parent = ref.random_tree(rng, N, max_children=int(rng.integers(2, 6)))
        if len(parent) - N > 5:
            continue
        for n_states in (2, 4):
            leaves = rng.integers(0, n_states, (N, 40))
            score, state, changed = ref.hartigan(parent, leaves, n_states)
            assert (score == brute_force(parent, leaves, n_states)).all()
            # the reconstruction is an optimal assignment: its changes equal the score, character by character
            assert (changed.sum(axis=0) == score).all()
            assert (state[:N] == leaves).all() and not changed[-1].any()


def test_reference_hand_worked_cases():
    A, Cc = 0, 1
    # polytomy (A, A, C, C): one node, four children; m = 2, so 4 - 2 = 2
    s, _, _ = ref.hartigan(np.array([4, 4, 4, 4, NONE], np.uint32), np.array([[A], [A], [Cc], [Cc]]), 4)
    assert s.tolist() == [2]
    # ((A, C), (A, C)) scores 2; ((A, A), (C, C)) scores 1
    t = np.array([4, 4, 5, 5, 6, 6, NONE], np.uint32)
    s, _, ch = ref.hartigan(t, np.array([[A], [Cc], [A], [Cc]]), 4)
    assert s.tolist() == [2] and int(ch.sum()) == 2
    s, st, ch = ref.hartigan(t, np.array([[A], [A], [Cc], [Cc]]), 4)
    assert s.tolist() == [1]
    # root {A, C} takes A; node 5 ({C}) changes, node 4 ({A}) does not
    assert st[:, 0].tolist() == [A, A, Cc, Cc, A, Cc, A] and ch[:, 0].tolist() == [0, 0, 0, 0, 0, 1, 0]
    # N = 1: the leaf is the root, nothing changes
    s, _, ch = ref.hartigan(np.array([NONE], np.uint32), np.array([[2, 3]]), 4)
    assert s.tolist() == [0, 0] and not ch.any()


def test_reference_summary_and_gains_losses():
    # ((0, 1), (2, 3), 4): polytomy root over two cherries and a leaf
    parent = np.array([5, 5, 6, 6, 7, 7, 7, NONE], np.uint32)
    pres = np.array([[1, 0], [1, 0], [0, 0], [0, 1], [1, 1]], np.uint8)
    s, sc, gains, losses = ref.gene_parsimony(parent, pres)
    # gene 0: root children {1}, {0}, {1} -> m = 2 (present), 1 change (node 6 loses); gene 1: cherry 6 = {0, 1}
    # costs 1, root children {0}, {0, 1}, {1} -> n = (2, 2), m = 2, 1 more: score 2
    assert sc.tolist() == [1, 2]
    assert s == (2, 2, 3, 2, 2 + 2, 1)
    assert int(gains.sum() + losses.sum()) == int(sc.sum())
    assert losses.tolist()[6] == 1 and gains.tolist()[3] == 1 and gains.tolist()[4] == 1


def test_reference_table_each_rule_once():
    good = np.array([3, 3, 4, 4, NONE], np.uint32)       # N = 3: ((0, 1), 2)
    ref.validate(good, 3)
    cases = {
        "fewer nodes than leaves": (good[:2], 3),
        "more than 2N - 1 nodes": (np.array([3, 3, 4, 4, 5, NONE], np.uint32), 3),
        "root not last": (np.array([3, 3, 4, NONE, 3], np.uint32), 3),
        "parent not above child": (np.array([3, 3, 4, 2, NONE], np.uint32), 3),
        "leaf as parent": (np.array([2, 3, 4, 4, NONE], np.uint32), 3),
        "parent out of range": (np.array([3, 3, 9, 4, NONE], np.uint32), 3),
        "internal node with one child": (np.array([4, 4, 3, 4, NONE], np.uint32), 3),
    }
    for t, N in cases.values():
        with pytest.raises(ValueError):
            ref.validate(t, N)
    ref.validate(np.array([NONE], np.uint32), 1)           # N = 1: the single leaf is the root


def test_indices_match_reference_including_nan():
    class S:
        pass
    for s in [(10, 4, 12, 6, 30, 2), (5, 0, 0, 0, 0, 0), (3, 1, 2, 2, 2, 0), (7, 3, 0, 0, 5, 0), (1, 1, 9, 1, 1, 1),
              (2**40, 7, 2**35 + 3, 2**33, 2**36, 5)]:
        o = S()
        for f, v in zip(PARSIMONY_FIELDS, s):
            setattr(o, f, v)
        got = parsimony_indices(o)
        want = ref.indices(s)
        for g, w in zip(got, want):
            assert (math.isnan(g) and math.isnan(w)) or g == w, (s, got, want)


def test_clades_first_leaf_and_size():
    parent = np.array([5, 5, 6, 6, 7, 7, 7, NONE], np.uint32)
    first, below = clades(parent, 5)
    assert first.tolist() == [0, 1, 2, 3, 4, 0, 2, 0] and below.tolist() == [1, 1, 1, 1, 1, 2, 2, 5]


def test_parsimony_symbols_exported_and_declared():
    L = C.CDLL(_ffi.build())
    header = open(os.path.join(ROOT, "include", "pansim_b200.h")).read()
    for name in SYMBOLS:
        assert hasattr(L, name) and name in _ffi.EXPORTED
        assert re.search(r"\bint\s+" + name + r"\(", header), name
    assert hasattr(L, "pansim_parsimony_indices") and "pansim_parsimony_indices" in _ffi.EXPORTED
    assert "typedef struct { uint64_t characters, variable, tree_length, min_changes, max_changes, homoplastic; } pansim_parsimony;" in header
    assert C.sizeof(_ffi.Parsimony) == 48
    assert "PANSIM_PARSIMONY_SCRATCH_MB" in open(os.path.join(ROOT, "DESIGN.md")).read()


def test_print_parsimony_flag_in_both_hosts():
    from pansim_b200.__main__ import build_parser
    assert vars(build_parser().parse_args([]))["print_parsimony"] is False
    assert vars(build_parser().parse_args(["--print_parsimony"]))["print_parsimony"] is True
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)
    r = subprocess.run([os.path.join(ROOT, "pansim_b200", "pansim"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--print_parsimony\n" in r.stdout


@pytest.mark.skipif(not os.path.exists(NVCC), reason="no nvcc")
def test_parsimony_kernels_have_no_spills_and_no_stack(tmp_path):
    src = tmp_path / "k.cu"
    src.write_text('#include "parsimony.cuh"\n'
                   "template __global__ void pansim::parsimony_kernel<4>(pansim::ParsimonyArgs);\n"
                   "template __global__ void pansim::parsimony_kernel<2>(pansim::ParsimonyArgs);\n")
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-cubin",
                        "-I", CSRC, "-o", str(tmp_path / "k.cubin"), str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    info = dict(re.findall(r"Compiling entry function '(\w+)'.*?\n.*?\n\s*(\d+ bytes stack frame, \d+ bytes spill stores, "
                           r"\d+ bytes spill loads)", r.stderr))
    ps = {k: v for k, v in info.items() if "parsimony" in k}
    assert len(ps) == 2, info
    assert all(v == "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" for v in ps.values()), ps
