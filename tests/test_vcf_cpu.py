"""Core-genome VCF without a device: the new symbols are exported, bound and declared, both command lines accept
--print_vcf, and the VCF kernels compile for sm_100a without spills."""
import ctypes as C
import os
import re
import subprocess

import pytest

from pansim_b200 import _ffi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SYMBOLS = ("pansim_write_core_vcf", "pansim_group_write_core_vcf", "pansim_core_vcf_kernel_ms")


def test_vcf_symbols_exported_and_declared():
    L = C.CDLL(_ffi.build())
    header = open(os.path.join(ROOT, "include", "pansim_b200.h")).read()
    for name in SYMBOLS:
        assert hasattr(L, name) and name in _ffi.EXPORTED
        assert re.search(r"\bint\s+" + name + r"\(", header), name
    assert "int pansim_write_core_vcf(pansim_ctx *ctx, const char *path, int with_header, uint64_t *bytes_out);" in header
    assert "int pansim_group_write_core_vcf(pansim_group *g, const char *path, uint64_t *bytes_out);" in header


def test_print_vcf_flag_in_both_hosts():
    from pansim_b200.__main__ import build_parser
    assert vars(build_parser().parse_args(["--print_vcf"]))["print_vcf"] is True
    assert vars(build_parser().parse_args([]))["print_vcf"] is False
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)
    r = subprocess.run([os.path.join(ROOT, "pansim_b200", "pansim"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--print_vcf" in r.stdout


NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


@pytest.mark.skipif(not os.path.exists(NVCC), reason="no nvcc")
def test_vcf_kernels_have_no_spills(tmp_path):
    src = tmp_path / "vcf.cu"
    src.write_text('#include "vcf.cuh"\n')
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-cubin",
                        "-I", os.path.join(ROOT, "pansim_b200", "csrc"), "-o", str(tmp_path / "vcf.cubin"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    kernels = re.findall(r"Compiling entry function '(\w+)'", r.stderr)
    assert len(kernels) == 5 and all("vcf_" in k for k in kernels), r.stderr
    frames = re.findall(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", r.stderr)
    assert len(frames) == 5 and all(f == ("0", "0", "0") for f in frames), r.stderr
