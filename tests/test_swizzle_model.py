"""Byte placement of bitmma_mainloop<KB> (bitmma.cuh) against the canonical shared-memory swizzles of the
tensor-core operand layouts (CuTe Swizzle<B, M, S>: the B address bits from bit M + S up are XOR-ed into the B bits
from bit M up; K-major SWIZZLE_128B = Swizzle<3,4,3>, SWIZZLE_64B = Swizzle<2,4,3>; tile base aligned to 1 KiB). CPU only."""
import pytest


def canonical(offset, bits):
    return offset ^ (((offset >> 7) & ((1 << bits) - 1)) << 4)


def kernel_address(row, k, kb):
    """dst + ((chunk << 4) ^ sw) with dst = tile + row * KB, sw = (row & 7) << 4 (KB = 128) or ((row >> 1) & 3) << 4 (KB = 64)."""
    sw = ((row & 7) if kb == 128 else ((row >> 1) & 3)) << 4
    return row * kb + (((k // 16) << 4) ^ sw) + k % 16


@pytest.mark.parametrize("kb,bits", [(128, 3), (64, 2)])
def test_expansion_writes_the_canonical_swizzle(kb, bits):
    seen = set()
    for row in range(128):
        for k in range(kb):
            a = kernel_address(row, k, kb)
            assert a == canonical(row * kb + k, bits), (row, k)
            seen.add(a)
    assert seen == set(range(128 * kb))          # a permutation of the tile


def test_gene_to_byte_permutation_covers_every_gene_once():
    """Word q of a row's stage goes to chunks 2q and 2q + 1; u32 t of the two chunks holds (v >> t) & 0x01010101,
    i.e. byte 4t + j of the 32 = bit t + 8j of the word: every gene exactly once, the same for both operands."""
    for v_bit in range(32):
        v = 1 << v_bit
        out = []
        for t in range(8):
            u = (v >> t) & 0x01010101
            out += [(u >> (8 * j)) & 0xFF for j in range(4)]
        assert sum(out) == 1 and out.index(1) == 4 * (v_bit % 8) + v_bit // 8
