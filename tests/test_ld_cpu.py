"""Core-genome LD without a device: the symbols are exported, bound and declared, pansim_ld_mean_r2 is the header's
formula, both command lines accept the --print_ld flags, ld.cuh compiles for sm_100a without spills with a tcgen05 MMA
in the pair kernel, and a hand-derived example of the numpy reference."""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np
import pytest

from ld_reference import np_ld_from_derived
from pansim_b200 import _ffi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SYMBOLS = ("pansim_core_ld", "pansim_group_core_ld", "pansim_core_ld_kernel_ms", "pansim_ld_mean_r2")


def test_ld_symbols_exported_and_declared():
    L = C.CDLL(_ffi.build())
    header = open(os.path.join(ROOT, "include", "pansim_b200.h")).read()
    for name in SYMBOLS:
        assert hasattr(L, name) and name in _ffi.EXPORTED
        assert re.search(r"\b(int|double)\s+" + name + r"\(", header), name
    assert "typedef struct { uint32_t max_dist, bin_width, min_minor; } pansim_ld_params;" in header
    assert "typedef struct { uint64_t pairs, four_gamete, r2_hi, r2_lo; } pansim_ld_bin;" in header


@pytest.mark.parametrize("pairs,hi,lo", [(0, 0, 0), (0, 5, 7), (1, 0, 1 << 32), (3, 5, 7), (12345, 2, 2**64 - 1),
                                         (2**40, 2**31, 2**63 + 12345)])
def test_mean_r2_is_the_header_formula(pairs, hi, lo):
    _ffi.lib()
    got = _ffi.lib().pansim_ld_mean_r2(C.byref(_ffi.LdBin(pairs, 0, hi, lo)))
    if pairs == 0:
        assert math.isnan(got)
    else:
        assert got == (math.ldexp(float(hi), 32) + math.ldexp(float(lo), -32)) / float(pairs)


def test_print_ld_flags_in_both_hosts():
    from pansim_b200.__main__ import build_parser
    ns = vars(build_parser().parse_args([]))
    assert (ns["print_ld"], ns["ld_max_dist"], ns["ld_bin_width"], ns["ld_min_minor"]) == (False, 10000, 100, 1)
    ns = vars(build_parser().parse_args(["--print_ld", "--ld_max_dist", "7", "--ld_bin_width", "3", "--ld_min_minor", "2"]))
    assert (ns["print_ld"], ns["ld_max_dist"], ns["ld_bin_width"], ns["ld_min_minor"]) == (True, 7, 3, 2)
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)
    r = subprocess.run([os.path.join(ROOT, "pansim_b200", "pansim"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--print_ld" in r.stdout
    for flag, default in (("ld_max_dist", 10000), ("ld_bin_width", 100), ("ld_min_minor", 1)):
        assert f"--{flag} <{flag}> [default: {default}]" in r.stdout


NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


@pytest.mark.skipif(not os.path.exists(NVCC), reason="no nvcc")
def test_ld_kernels_have_no_spills_and_use_tcgen05(tmp_path):
    src = tmp_path / "ld.cu"
    src.write_text('#include "ld.cuh"\n')
    cubin = str(tmp_path / "ld.cubin")
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-cubin",
                        "-I", os.path.join(ROOT, "pansim_b200", "csrc"), "-o", cubin, str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    info = dict(re.findall(r"Compiling entry function '(\w+)'.*?\n.*?\n\s*(\d+ bytes stack frame, \d+ bytes spill stores, \d+ bytes spill loads)",
                           r.stderr))
    ld = {k: v for k, v in info.items() if "ld_" in k and "vcf" not in k}
    assert len(ld) == 5, r.stderr
    assert all(v == "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" for v in ld.values()), ld
    pair = next(k for k in ld if "ld_pair_kernel" in k)
    sass = subprocess.run([os.path.join(os.path.dirname(NVCC), "cuobjdump"), "-sass", "-fun", pair, cubin],
                          capture_output=True, text=True).stdout
    assert re.search(r"\bUTC\w*MMA", sass) and "LDTM" in sass
    assert not re.search(r"\b[HI]MMA\b", sass)


def test_reference_hand_derived_example():
    # 5 rows x 4 sites, derived counts a = 3, 2, 3, 2, so a (n - a) = 6 and inv = 1/6 at every site.
    der = np.array([[1, 1, 0, 0],
                    [1, 1, 1, 0],
                    [1, 0, 1, 0],
                    [0, 0, 0, 1],
                    [0, 0, 1, 1]], bool)
    # pair   d  c   D = 5c - a_i a_j   r2      four gametes
    # (0,1)  1  2    4                 16/36   no  (a_j - c = 0)
    # (0,2)  2  2    1                  1/36   yes
    # (0,3)  3  0   -6                  1      no  (c = 0)
    # (1,2)  1  1   -1                  1/36   yes
    # (1,3)  2  0   -4                 16/36   no
    # (2,3)  1  1   -1                  1/36   yes
    # max_dist 3, bin width 2: bin 0 = d 1..2, bin 1 = d 3. q = rint(r2 2^32): 16/36 -> 1908874354, 1/36 -> 119304647.
    pairs, fg, r2, used = np_ld_from_derived(der, 3, 2, 1)
    assert used == 4
    assert list(pairs) == [5, 1] and list(fg) == [3, 0]
    assert r2 == [2 * 1908874354 + 3 * 119304647, 1 << 32]
    # min_minor 3 leaves no site used (min(a, n - a) <= 2); a window of 1 keeps the three d = 1 pairs
    assert np_ld_from_derived(der, 3, 2, 3)[3] == 0
    pairs, fg, r2, _ = np_ld_from_derived(der, 1, 1, 1)
    assert list(pairs) == [3] and list(fg) == [2] and r2 == [1908874354 + 2 * 119304647]
