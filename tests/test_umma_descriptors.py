"""tcgen05 descriptors of the bit-matrix product pipeline (bitmma.cuh), decoded field by field on the host (no GPU).

Instruction descriptor (kind::i8) and shared-memory matrix descriptor layouts as in CUTLASS
cute/arch/mma_sm100_desc.hpp (InstrDescriptor, SmemDescriptor): a silent edit of one constant would make the
tensor core read garbage, which only the GPU parity tests would notice. Also what the compiler makes of the
competition term's kernel (select.cuh): registers, spills and tensor-core instructions."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"

SRC = r'''
#include <cstdio>
#include "bitmma.cuh"
int main()
{
    using namespace pansim;
    printf("%u %u %u %zu %zu %d %d\n", UM_IDESC, UbCfg<128>::DESC_HI, UbCfg<64>::DESC_HI, UbCfg<128>::smem_bytes(),
           UbCfg<64>::smem_bytes(), UB_THREADS, UM_TILE);
    return 0;
}
'''


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_bitmma_descriptor_fields(tmp_path):
    src = tmp_path / "desc.cu"
    src.write_text(SRC)
    exe = str(tmp_path / "desc")
    subprocess.run([NVCC, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-I", os.path.join(ROOT, "pansim_b200", "csrc"),
                    "-o", exe, str(src)], check=True, capture_output=True)
    idesc, hi128, hi64, smem128, smem64, threads, tile = map(int, subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split())
    # instruction descriptor: dense, no saturation, D = s32 (2 at bits 4-5), A = B = u8 (0 at bits 7-9 / 10-12), no negation,
    # both operands K-major (bits 15, 16 = 0), N >> 3 at bits 17-22, M >> 4 at bits 24-28, no shift
    assert idesc & 0xF == 0 and (idesc >> 4) & 3 == 2
    assert (idesc >> 7) & 7 == 0 and (idesc >> 10) & 7 == 0 and (idesc >> 13) & 0xF == 0
    assert (idesc >> 17) & 0x3F == tile >> 3 and (idesc >> 24) & 0x1F == tile >> 4 and idesc >> 29 == 0
    assert tile == 128
    # matrix descriptor, high word: stride between 8-row groups in 16-byte units (bits 0-13), version 1 (bits 14-15),
    # base offset 0, layout (bits 29-31): 2 = SWIZZLE_128B, 4 = SWIZZLE_64B
    for hi, row_bytes, layout in ((hi128, 128, 2), (hi64, 64, 4)):
        assert hi & 0x3FFF == 8 * row_bytes // 16
        assert (hi >> 14) & 3 == 1 and (hi >> 16) & 0x1FFF == 0 and hi >> 29 == layout
    # shared memory: 1 KiB alignment slack + operand stages + mbarriers + the tensor-memory address slot
    assert smem128 == 1024 + 2 * 4 * 128 * 128 + 9 * 8 + 16
    assert smem64 == 1024 + 2 * 3 * 128 * 64 + 7 * 8 + 16 and smem64 <= 56 * 1024
    assert threads == 288


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_competition_kernel_is_tcgen05_without_spills(tmp_path):
    """The intersection counts run on tcgen05 (UTC*MMA, tcgen05.ld = LDTM) in at most 71 registers with no spills, and
    no kernel of select.cuh falls back to warp-level mma.sync (HMMA / IMMA)."""
    src = tmp_path / "select.cu"
    src.write_text('#include "select.cuh"\n')
    cubin = str(tmp_path / "select.cubin")
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-cubin",
                        "-I", os.path.join(ROOT, "pansim_b200", "csrc"), "-o", cubin, str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    info = re.search(r"Compiling entry function '(\w*acc_inter_umma_bits_kernel\w*)'.*?\n.*?\n\s*(\d+) bytes stack frame, "
                     r"(\d+) bytes spill stores, (\d+) bytes spill loads\n.*?Used (\d+) registers", r.stderr)
    assert info, r.stderr
    name, stack, stores, loads, regs = info.group(1), *map(int, info.groups()[1:])
    assert (stack, stores, loads) == (0, 0, 0) and regs <= 71, info.group(0)
    cuobjdump = os.path.join(os.path.dirname(NVCC), "cuobjdump")
    sass = subprocess.run([cuobjdump, "-sass", "-fun", name, cubin], capture_output=True, text=True).stdout
    assert re.search(r"\bUTC\w*MMA", sass) and "LDTM" in sass
    every = subprocess.run([cuobjdump, "-sass", cubin], capture_output=True, text=True).stdout
    assert "Function :" in every and not re.search(r"\b[HI]MMA\b", every)
