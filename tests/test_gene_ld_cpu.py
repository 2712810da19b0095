"""Accessory-gene linkage without a device: the symbols are exported, bound and declared with their structs, both
command lines accept the --print_gene_ld flags, gene_ld.cuh compiles for sm_100a without spills with a tcgen05 MMA in
the pair kernel, ld_pair_kernel keeps its registers after sharing its pipeline, and a hand-derived example of the
numpy reference."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from gene_ld_reference import gene_groups, np_gene_ld
from pansim_b200 import _ffi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SYMBOLS = ("pansim_gene_ld", "pansim_group_gene_ld", "pansim_gene_ld_kernel_ms")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def test_gene_ld_symbols_exported_and_declared():
    L = C.CDLL(_ffi.build())
    header = open(os.path.join(ROOT, "include", "pansim_b200.h")).read()
    for name in SYMBOLS:
        assert hasattr(L, name) and name in _ffi.EXPORTED
        assert re.search(r"\bint\s+" + name + r"\(", header), name
    assert "typedef struct { uint32_t r2_bins, min_minor; } pansim_gene_ld_params;" in header
    assert "typedef struct { pansim_ld_bin ld; uint64_t associated, dissociated; } pansim_gene_ld_class;" in header
    assert C.sizeof(_ffi.GeneLdClass) == 48 and C.sizeof(_ffi.GeneLdParams) == 8


def test_print_gene_ld_flags_in_both_hosts():
    from pansim_b200.__main__ import build_parser
    ns = vars(build_parser().parse_args([]))
    assert (ns["print_gene_ld"], ns["gene_ld_bins"], ns["gene_ld_min_minor"]) == (False, 20, 1)
    ns = vars(build_parser().parse_args(["--print_gene_ld", "--gene_ld_bins", "7", "--gene_ld_min_minor", "3"]))
    assert (ns["print_gene_ld"], ns["gene_ld_bins"], ns["gene_ld_min_minor"]) == (True, 7, 3)
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)
    r = subprocess.run([os.path.join(ROOT, "pansim_b200", "pansim"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--print_gene_ld\n" in r.stdout
    for flag, default in (("gene_ld_bins", 20), ("gene_ld_min_minor", 1)):
        assert f"--{flag} <{flag}> [default: {default}]" in r.stdout


def _ptxas(tmp_path, header):
    src = tmp_path / "k.cu"
    src.write_text(f'#include "{header}"\n')
    cubin = str(tmp_path / "k.cubin")
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-cubin",
                        "-I", os.path.join(ROOT, "pansim_b200", "csrc"), "-o", cubin, str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    info = {k: (spill, regs) for k, spill, regs in
            re.findall(r"Compiling entry function '(\w+)'.*?\n.*?\n\s*(\d+ bytes stack frame, \d+ bytes spill stores, "
                       r"\d+ bytes spill loads)\n[^\n]*?Used (\d+ registers)", r.stderr)}
    return info, cubin


@pytest.mark.skipif(not os.path.exists(NVCC), reason="no nvcc")
def test_gene_ld_kernels_have_no_spills_and_use_tcgen05(tmp_path):
    info, cubin = _ptxas(tmp_path, "gene_ld.cuh")
    gl = {k: v for k, v in info.items() if "gene_ld_" in k}
    assert len(gl) == 4, info
    assert all(v[0] == "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" for v in gl.values()), gl
    pair = next(k for k in gl if "gene_ld_pair_kernel" in k)
    sass = subprocess.run([os.path.join(os.path.dirname(NVCC), "cuobjdump"), "-sass", "-fun", pair, cubin],
                          capture_output=True, text=True).stdout
    assert re.search(r"\bUTC\w*MMA", sass) and "LDTM" in sass
    assert not re.search(r"\b[HI]MMA\b", sass)


@pytest.mark.skipif(not os.path.exists(NVCC), reason="no nvcc")
def test_ld_pair_kernel_unchanged_by_the_shared_pipeline(tmp_path):
    # the register count and spill line ptxas gave ld_pair_kernel before its operand pipeline was shared
    info, _ = _ptxas(tmp_path, "ld.cuh")
    pair = next(v for k, v in info.items() if "ld_pair_kernel" in k)
    assert pair == ("0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads", "54 registers")


def test_reference_hand_derived_example():
    # 5 rows x 4 genes, presence counts a = 3, 2, 3, 2, so a (n - a) = 6 and inv = 1/6 for every gene;
    # genes 2 and 3 form group 1.
    pres = np.array([[1, 1, 0, 0],
                     [1, 1, 1, 0],
                     [1, 0, 1, 0],
                     [0, 0, 0, 1],
                     [0, 0, 1, 1]], bool)
    grp = gene_groups(4, 2, [0, 2], [2, 4])
    assert list(grp) == [0, 0, 1, 1]
    # pair   class  c   D = 5c - a_g a_h  r2     q            bin of 4  four gametes
    # (0,1)  0-0    2    4                16/36  1908874354   1         no  (a_h - c = 0)
    # (0,2)  0-1    2    1                 1/36   119304647   0         yes
    # (0,3)  0-1    0   -6                 1     2^32         3 (last)  no  (c = 0)
    # (1,2)  0-1    1   -1                 1/36   119304647   0         yes
    # (1,3)  0-1    0   -4                16/36  1908874354   1         no
    # (2,3)  1-1    1   -1                 1/36   119304647   0         yes
    r = np_gene_ld(pres, grp, 4, 1)
    assert r["pairs"] == [1, 4, 1] and r["four_gamete"] == [0, 2, 1]
    assert r["associated"] == [1, 1, 0] and r["dissociated"] == [0, 3, 1]
    assert r["r2_sum"] == [1908874354, 2 * 119304647 + (1 << 32) + 1908874354, 119304647]
    assert r["hist"].tolist() == [[0, 1, 0, 0], [2, 1, 0, 1], [1, 0, 0, 0]]
    assert list(r["genes_used"]) == [2, 2]
    # one bin holds every pair; min_minor 2 keeps every gene (min(a, n - a) = 2), 3 none
    r1 = np_gene_ld(pres, grp, 1, 2)
    assert r1["hist"].tolist() == [[1], [4], [1]] and r1["pairs"] == [1, 4, 1]
    r3 = np_gene_ld(pres, grp, 20, 3)
    assert r3["pairs"] == [0, 0, 0] and list(r3["genes_used"]) == [0, 0] and r3["hist"].sum() == 0
    # one compartment: every pair is 0-0
    r0 = np_gene_ld(pres, gene_groups(4, 1, [0], [4]), 4, 1)
    assert r0["pairs"] == [6, 0, 0] and r0["hist"].tolist()[0] == [3, 2, 0, 1]
