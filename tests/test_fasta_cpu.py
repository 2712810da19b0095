"""Core-genome FASTA without a device: the new symbols are exported, bound and declared, both command lines accept
--print_fasta and --print_snp_alignment, the FASTA kernels compile for sm_100a without spills or a stack frame, and
the numpy formatter reproduces a hand-worked example in both modes."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from fasta_reference import CODES, fasta_text, record_offset
from pansim_b200 import _ffi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DECLS = (
    "int pansim_write_core_fasta(pansim_ctx *ctx, const char *path, int snps_only, uint64_t *columns_out, "
    "uint64_t *const_counts /* [4] or NULL */, uint64_t *bytes_out);",
    "int pansim_export_core_fasta_rows(pansim_ctx *ctx, int snps_only, uint32_t row_begin, uint32_t row_end, char *out, "
    "uint64_t *columns_out);",
    "int pansim_group_write_core_fasta(pansim_group *g, const char *path, int snps_only, uint64_t *columns_out, "
    "uint64_t *const_counts, uint64_t *bytes_out);",
    "int pansim_core_fasta_kernel_ms(pansim_ctx *ctx, int snps_only, uint32_t repeats, float *site_ms, float *expand_ms, "
    "uint64_t *text_bytes);",
)


def test_fasta_symbols_exported_bound_and_declared():
    L = C.CDLL(_ffi.build())
    header = open(os.path.join(ROOT, "include", "pansim_b200.h")).read()
    bound = _ffi.lib()
    for decl in DECLS:
        name = re.match(r"int (\w+)\(", decl).group(1)
        assert hasattr(L, name) and name in _ffi.EXPORTED
        assert decl in header, name
        n_args = decl.count(",") + 1
        assert getattr(bound, name).restype is C.c_int and len(getattr(bound, name).argtypes) == n_args, name


def test_fasta_flags_in_both_hosts():
    from pansim_b200.__main__ import build_parser
    for flag in ("print_fasta", "print_snp_alignment"):
        assert vars(build_parser().parse_args(["--" + flag]))[flag] is True
        assert vars(build_parser().parse_args([]))[flag] is False
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)
    r = subprocess.run([os.path.join(ROOT, "pansim_b200", "pansim"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--print_fasta" in r.stdout and "--print_snp_alignment" in r.stdout


NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


@pytest.mark.skipif(not os.path.exists(NVCC), reason="no nvcc")
def test_fasta_kernels_have_no_spills(tmp_path):
    src = tmp_path / "fasta.cu"
    src.write_text('#include "fasta.cuh"\n')
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-cubin",
                        "-I", os.path.join(ROOT, "pansim_b200", "csrc"), "-o", str(tmp_path / "fasta.cubin"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    kernels = re.findall(r"Compiling entry function '(\w+)'", r.stderr)
    for name in ("fasta_site_kernel", "fasta_compact_kernel", "fasta_expand_kernel"):
        assert sum(name in k for k in kernels) == 1, r.stderr
    frames = re.findall(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", r.stderr)
    assert len(frames) == len(kernels) and all(f == ("0", "0", "0") for f in frames), r.stderr


def _onehot(rows):
    return CODES[np.array([["ACGT".index(ch) for ch in row] for row in rows])]


def test_reference_reproduces_the_hand_worked_example():
    # sites: 0 AAA, 1 CCG (2 letters), 2 GGG, 3 TTT, 4 ACG (3 letters), 5 AAA, 6 CCC, 7 GTA (3 letters), 8 TTT
    core = _onehot(["ACGTAACGT", "ACGTCACTT", "AGGTGACAT"])
    text, cols, const = fasta_text(core, snps_only=False)
    assert text == b">ind_0\nACGTAACGT\n>ind_1\nACGTCACTT\n>ind_2\nAGGTGACAT\n"
    assert cols == 9 and const.tolist() == [0, 0, 0, 0]
    text, cols, const = fasta_text(core, snps_only=True)
    assert text == b">ind_0\nCAG\n>ind_1\nCCT\n>ind_2\nGGA\n"
    assert cols == 3 and const.tolist() == [2, 1, 1, 2] and const.sum() + cols == 9
    # no polymorphic site: every record is ">ind_<i>\n\n"
    text, cols, const = fasta_text(_onehot(["ACGT", "ACGT"]), snps_only=True)
    assert text == b">ind_0\n\n>ind_1\n\n" and cols == 0 and const.tolist() == [1, 1, 1, 1]


@pytest.mark.parametrize("cols", [0, 1, 9, 1000])
def test_record_offsets_have_a_closed_form(cols):
    sizes = np.array([7 + len(str(i)) + cols for i in range(12000)], np.int64)
    starts = np.concatenate([[0], np.cumsum(sizes)])
    assert all(record_offset(i, cols) == starts[i] for i in list(range(0, 12001, 7)) + [9, 10, 11, 99, 100, 101, 999, 1000, 10000])
