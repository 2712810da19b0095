"""Core-genome diversity without a device: pansim_diversity_stats against a Python restatement in the same
summation order (bit for bit), the ABI of pansim_diversity, the CLI flags, and the kernel's register use."""
import ctypes as C
import math
import os
import re
import shutil
import subprocess

import pytest

import pansim_b200 as pb
from pansim_b200 import _ffi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAN = float("nan")


def restated_stats(seg: int, pair_diff_sum: int, n: int):
    """pi, theta_W and Tajima's D (1989) with a1, a2 summed for i = 1..n-1 in ascending order."""
    if n < 2:
        return NAN, NAN, NAN
    a1 = a2 = 0.0
    for i in range(1, n):
        x = float(i)
        a1 += 1.0 / x
        a2 += 1.0 / (x * x)
    pi = float(pair_diff_sum) / float(n * (n - 1) // 2)
    S = float(seg)
    tw = S / a1
    nn = float(n)
    b1 = (nn + 1.0) / (3.0 * (nn - 1.0))
    b2 = (2.0 * (nn * nn + nn + 3.0)) / (9.0 * nn * (nn - 1.0))
    c1 = b1 - 1.0 / a1
    c2 = b2 - (nn + 2.0) / (a1 * nn) + a2 / (a1 * a1)
    e1 = c1 / a1
    e2 = c2 / (a1 * a1 + a2)
    var = e1 * S + e2 * S * (S - 1.0)
    den = math.sqrt(var) if var >= 0.0 else NAN
    d = NAN if (seg == 0 or not den > 0.0) else (pi - tw) / den
    return pi, tw, d


def same_bits(a, b):
    return all((x == y) or (math.isnan(x) and math.isnan(y)) for x, y in zip(a, b))


CASES = [
    # (segregating, pair_diff_sum, N)
    (0, 0, 10),            # nothing segregates: pi = theta = 0, D = NaN
    (5, 21, 10),
    (1, 1, 2),             # N = 2: C(N,2) = 1, a1 = 1
    (3, 4, 3),
    (7, 0, 3),
    (1234, 987654, 100),
    (1, 1, 1000),
    (60000, 123456789012, 1000),
    (4_999_000, 10**15 + 7, 20000),
    (2**40, 2**62 + 12345, 70000),
]


@pytest.mark.parametrize("seg,pd,n", CASES)
def test_diversity_stats_bit_exact(seg, pd, n):
    d = pb.Diversity(sites=max(seg, 1), segregating=seg, multiallelic=0, pair_diff_sum=pd)
    got = pb.diversity_stats(d, n)
    want = restated_stats(seg, pd, n)
    assert same_bits(got, want), (got, want)


def test_diversity_stats_edge_values():
    assert all(math.isnan(x) for x in pb.diversity_stats(pb.Diversity(10, 3, 0, 5), 1))
    assert all(math.isnan(x) for x in pb.diversity_stats(pb.Diversity(10, 3, 0, 5), 0))
    pi, tw, d = pb.diversity_stats(pb.Diversity(10, 0, 0, 0), 50)
    assert pi == 0.0 and tw == 0.0 and math.isnan(d)
    # two sequences: pi = differing sites = S, a1 = 1, so D = 0 whenever it is defined
    pi, tw, d = pb.diversity_stats(pb.Diversity(100, 7, 0, 7), 2)
    assert pi == 7.0 and tw == 7.0
    # a site where one of n individuals carries a singleton: pi = (n-1)/C(n,2) = 2/n < theta_W = 1/a1 -> D < 0
    n = 30
    pi, tw, d = pb.diversity_stats(pb.Diversity(100, 1, 0, n - 1), n)
    assert pi == 2.0 / n and d < 0.0


def test_diversity_symbols_and_struct_size(tmp_path):
    L = C.CDLL(_ffi.build())
    for name in ("pansim_core_allele_counts", "pansim_core_diversity", "pansim_run_generations_diversity",
                 "pansim_diversity_stats", "pansim_group_core_diversity", "pansim_group_run_generations_diversity"):
        assert hasattr(L, name) and name in _ffi.EXPORTED
    assert C.sizeof(_ffi.Diversity) == 32
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "sz.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "pansim_b200.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu\\n", sizeof(pansim_diversity), offsetof(pansim_diversity, sites),'
                   ' offsetof(pansim_diversity, segregating), offsetof(pansim_diversity, multiallelic),'
                   ' offsetof(pansim_diversity, pair_diff_sum));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(_ffi.Diversity)] + [getattr(_ffi.Diversity, f).offset for f, _ in _ffi.Diversity._fields_]
    assert got == want


def test_print_diversity_flag_in_both_hosts():
    from pansim_b200.__main__ import build_parser
    ns = vars(build_parser().parse_args(["--print_diversity"]))
    assert ns["print_diversity"] is True
    assert vars(build_parser().parse_args([]))["print_diversity"] is False
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)
    r = subprocess.run([os.path.join(ROOT, "pansim_b200", "pansim"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--print_diversity" in r.stdout


NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


@pytest.mark.skipif(not os.path.exists(NVCC), reason="no nvcc")
def test_diversity_kernel_has_no_spills(tmp_path):
    src = tmp_path / "dv.cu"
    src.write_text('#include "diversity.cuh"\n'
                   "template __global__ void pansim::diversity_kernel<false, false>(pansim::DiversityArgs);\n"
                   "template __global__ void pansim::diversity_kernel<false, true>(pansim::DiversityArgs);\n"
                   "template __global__ void pansim::diversity_kernel<true, false>(pansim::DiversityArgs);\n")
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-cubin",
                        "-I", os.path.join(ROOT, "pansim_b200", "csrc"), "-o", str(tmp_path / "dv.cubin"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", r.stderr)
    assert len(spills) == 3, r.stderr
    assert all(s == ("0", "0") for s in spills), r.stderr
