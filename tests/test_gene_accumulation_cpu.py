"""Pangenome accumulation without a device: the symbols are exported, bound and declared, both command lines accept
the --print_gene_accumulation flags, pangenome.cuh compiles for sm_100a without spills or stack, the numpy Philox
restatement equals philox4x32_10 of common.cuh, a hand-derived example of the reference, and the gene classes at
Roary's threshold boundaries."""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np
import pytest

from gene_accumulation_reference import ORDER_TAG, np_classes, np_curves, np_orders, np_spectrum, philox4x32_10
from pansim_b200 import _ffi
from pansim_b200.population import pangenome_classes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SYMBOLS = ("pansim_gene_accumulation", "pansim_group_gene_accumulation", "pansim_gene_accumulation_kernel_ms",
           "pansim_gene_spectrum", "pansim_group_gene_spectrum")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CSRC = os.path.join(ROOT, "pansim_b200", "csrc")


def test_gene_accumulation_symbols_exported_and_declared():
    L = C.CDLL(_ffi.build())
    header = open(os.path.join(ROOT, "include", "pansim_b200.h")).read()
    for name in SYMBOLS:
        assert hasattr(L, name) and name in _ffi.EXPORTED
        assert re.search(r"\bint\s+" + name + r"\(", header), name
    assert hasattr(L, "pansim_pangenome_classes") and "pansim_pangenome_classes" in _ffi.EXPORTED
    assert re.search(r"\bvoid\s+pansim_pangenome_classes\(const uint64_t \*spectrum, uint32_t pop_size, uint64_t out\[5\]\)", header)
    assert f"#define PANSIM_GENE_ACC_ORDER_TAG 0x{ORDER_TAG:08X}u" in header
    assert "#define PANSIM_GENE_ACC_MAX_PERMS 10000u" in header


def test_print_gene_accumulation_flags_in_both_hosts():
    from pansim_b200.__main__ import build_parser
    ns = vars(build_parser().parse_args([]))
    assert (ns["print_gene_accumulation"], ns["gene_accumulation_perms"]) == (False, 100)
    ns = vars(build_parser().parse_args(["--print_gene_accumulation", "--gene_accumulation_perms", "7"]))
    assert (ns["print_gene_accumulation"], ns["gene_accumulation_perms"]) == (True, 7)
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)
    r = subprocess.run([os.path.join(ROOT, "pansim_b200", "pansim"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--print_gene_accumulation\n" in r.stdout
    assert "--gene_accumulation_perms <gene_accumulation_perms> [default: 100]" in r.stdout


@pytest.mark.skipif(not os.path.exists(NVCC), reason="no nvcc")
def test_pangenome_kernels_have_no_spills_and_no_stack(tmp_path):
    src = tmp_path / "k.cu"
    src.write_text('#include "pangenome.cuh"\n'
                   "template __global__ void pansim::pg_order_kernel<true>(pansim::PgOrderArgs);\n"
                   "template __global__ void pansim::pg_order_kernel<false>(pansim::PgOrderArgs);\n")
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-cubin",
                        "-I", CSRC, "-o", str(tmp_path / "k.cubin"), str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    info = dict(re.findall(r"Compiling entry function '(\w+)'.*?\n.*?\n\s*(\d+ bytes stack frame, \d+ bytes spill stores, "
                           r"\d+ bytes spill loads)", r.stderr))
    pg = {k: v for k, v in info.items() if "pg_" in k}
    assert len(pg) == 6, info                  # order (both paths), summary, walk, curves, spectrum
    assert all(v == "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" for v in pg.values()), pg


@pytest.mark.skipif(not os.path.exists(NVCC), reason="no nvcc")
def test_numpy_philox_equals_common_cuh(tmp_path):
    # a host-only program: philox4x32_10 of common.cuh is __host__ __device__, so no device is needed
    ctrs = [(0, 0, 0, 0), (1, 2, 3, 4), (0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF), (17, 99, 0, ORDER_TAG),
            (123456, 7, 0, ORDER_TAG), (0x80000000, 0x12345678, 0x9ABCDEF0, 0x0F0F0F0F)]
    keys = [(0, 0), (1, 0), (0xDEADBEEF, 0x01234567), (0xFFFFFFFF, 0xFFFFFFFF)]
    lines = "".join(f"    pr(make_uint4({a}u, {b}u, {c}u, {d}u), make_uint2({k0}u, {k1}u));\n"
                    for (a, b, c, d) in ctrs for (k0, k1) in keys)
    src = tmp_path / "philox.cu"
    src.write_text('#include <cstdio>\n#include "common.cuh"\nusing namespace pansim;\n'
                   'static void pr(uint4 c, uint2 k) { uint4 r = philox4x32_10(c, k); printf("%u %u %u %u\\n", r.x, r.y, r.z, r.w); }\n'
                   "int main() {\n" + lines + "    return 0;\n}\n")
    exe = str(tmp_path / "philox")
    r = subprocess.run([NVCC, "-std=c++17", "-I", CSRC, "-o", exe, str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = [tuple(int(x) for x in line.split()) for line in subprocess.run([exe], capture_output=True, text=True,
                                                                             check=True).stdout.splitlines()]
    want = [tuple(int(w) for w in philox4x32_10(c, k)) for c in ctrs for k in keys]
    assert got == want


def test_reference_orders_are_fisher_yates():
    # the vectorised draw equals a plain loop over one order at a time
    seed, P, N = 0x1234_5678_9ABC, 5, 37
    got = np_orders(seed, P, N)
    for p in range(P):
        o = list(range(N))
        for i in range(N - 1, 0, -1):
            r = int(philox4x32_10((i, p, 0, ORDER_TAG), (seed & 0xFFFFFFFF, seed >> 32))[0])
            j = (r * (i + 1)) >> 32
            o[i], o[j] = o[j], o[i]
        assert got[p].tolist() == o
    assert sorted(got[0].tolist()) == list(range(N)) and not np.array_equal(got, np_orders(seed + 1, P, N))
    assert np_orders(3, 2, 1).tolist() == [[0], [0]]


def test_reference_hand_derived_example():
    # 4 rows x 5 genes, c0 = 2, order 2, 0, 3, 1
    pres = np.array([[1, 1, 0, 0, 0],
                     [1, 0, 1, 0, 0],
                     [1, 1, 1, 1, 0],
                     [0, 0, 0, 0, 1]], bool)
    # k  row  genes      seen once  in all   pan  core  new  unique
    # 1  2    0,1,2,3    0,1,2,3    0,1,2,3  6    6     6    6 (every gene is unique at k = 1)
    # 2  0    0,1        2,3        0,1      6    4     0    2
    # 3  3    4          2,3,4      -        7    2     1    3
    # 4  1    0,2        3,4        -        7    2     0    2
    pan, core, new, unique = np_curves(pres, [[2, 0, 3, 1]], 2)
    assert pan.tolist() == [[6, 6, 7, 7]] and core.tolist() == [[6, 4, 2, 2]]
    assert new.tolist() == [[6, 0, 1, 0]] and unique.tolist() == [[6, 2, 3, 2]]
    assert (np.cumsum(new, axis=1) == pan).all()
    # a = 3, 2, 2, 1, 1; the two c0 genes in bin 4
    spec = np_spectrum(pres, 2)
    assert spec.tolist() == [0, 2, 2, 1, 2]
    # N = 4: only a = 4 is core (400 >= 396); a = 3 (300 < 380) down to a = 1 (100 >= 60) are shell
    assert np_classes(spec, 4) == (2, 0, 5, 0, 7) == pangenome_classes(spec, 4)


# Hand-made classes (0 core, 1 soft core, 2 shell, 3 cloud) at a = ceil(0.99 N) - 1, ceil(0.99 N), ceil(0.95 N),
# ceil(0.15 N) and one row below the last three:
#   N = 7:     100 a against 693 / 665 / 105; ceil(0.95 * 7) = ceil(0.99 * 7) = 7
#   N = 100:   against 9 900 / 9 500 / 1 500
#   N = 1 000: against 99 000 / 95 000 / 15 000
BOUNDARY_CLASSES = {
    7: {6: 2, 7: 0, 2: 2, 1: 3, 5: 2},
    100: {98: 1, 99: 0, 95: 1, 15: 2, 97: 1, 94: 2, 14: 3},
    1000: {989: 1, 990: 0, 950: 1, 150: 2, 988: 1, 949: 2, 149: 3},
}


@pytest.mark.parametrize("N", sorted(BOUNDARY_CLASSES))
def test_classes_exact_at_roary_boundaries(N):
    for a, cls in BOUNDARY_CLASSES[N].items():
        spec = np.zeros(N + 1, np.uint64)
        spec[a] = 3
        want = [0, 0, 0, 0, 3]
        want[cls] = 3
        assert pangenome_classes(spec, N) == tuple(want) == np_classes(spec, N), (N, a)
    assert {math.ceil(0.99 * N) - 1, math.ceil(0.99 * N), math.ceil(0.95 * N), math.ceil(0.15 * N)} <= set(BOUNDARY_CLASSES[N])
    # every bin at once; bin 0 (genes no row carries) is not counted
    spec = np.ones(N + 1, np.uint64)
    want = {7: (1, 0, 5, 1, 7), 100: (2, 4, 80, 14, 100), 1000: (11, 40, 800, 149, 1000)}[N]
    assert pangenome_classes(spec, N) == want == np_classes(spec, N)
